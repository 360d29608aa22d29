"""The learner path on the GPU: actor / critic networks, parameter-noise
exploration, replay ring, critic fit and actor policy-gradient step.

Three layers, all ending in launches of the CUDA library (C ABI:
include/skillshot_b200.h); there is no CPU path.

* :class:`ActorCritic` -- the two networks of SkillshotLearner.model_define_actor /
  model_define_critic (SkillshotLearner.py:70-121) as flat float32 parameter
  vectors with their tf.keras Adam state and (DDPG) target copies, and the batched
  device operations on them.
* :class:`ReplayRing` -- device-resident transitions.
* :class:`SkillshotLearner` -- the reference's class surface (same method names,
  argument meaning and attribute-style hyper-parameters) over one SkillshotGame.
* :class:`SelfPlayTrainer` -- the same loop for many envs at once: rollout of N
  games with the shared actor, replay, sharded update with one gradient all-reduce.
"""
from __future__ import annotations

import ctypes
import math
import os
from typing import Optional

import numpy as np
import torch

from . import _lib
from ._lib import check, lib
from .game import FEATURE_KEYS, REWARD_MODES, SkillshotEnvs, SkillshotGame
from .match import Match, actor_vector

A_N, C_N = _lib.ACTOR_PARAMS, _lib.CRITIC_PARAMS
ACTOR_SHAPES = [(12, 256), (256,), (256, 128), (128,), (128, 2), (2,)]       # Keras get_weights() order
CRITIC_SHAPES = [(12, 256), (256,), (258, 128), (128,), (128, 1), (1,)]


def _ptr(t):
    return None if t is None else t.data_ptr()


def _stream(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _f32(x, device, shape=None):
    if not torch.is_tensor(x):
        x = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32))
    x = x.to(device=device, dtype=torch.float32).contiguous()
    return x if shape is None else x.reshape(shape)


def split_params(flat, shapes):
    """Views of a flat parameter vector in Keras get_weights() order."""
    out, o = [], 0
    for s in shapes:
        n = int(np.prod(s))
        out.append(flat[o:o + n].reshape(s))
        o += n
    return out


def shard_info(n_local: int, group=None):
    """(world, n_global, row_offset) of a batch sharded evenly over the ranks of `group`
    (None: not distributed; True: the default group).  Rank r owns global rows
    [r * n_local, (r + 1) * n_local): the critic's mean divides by n_global and Philox dropout is
    keyed by the global row, so a sharded update equals the single-GPU update of the whole batch."""
    if group is None:
        return 1, n_local, 0
    import torch.distributed as dist
    g = None if group is True else group
    world, rank = dist.get_world_size(g), dist.get_rank(g)
    return world, n_local * world, rank * n_local


def allreduce_sum(t: torch.Tensor, group=None):
    """The one exchange step of a sharded update: sum the flat gradient over ranks (NCCL on GPUs)."""
    if group is None:
        return t
    import torch.distributed as dist
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=None if group is True else group)
    return t


def check_process_group(group):
    """ValueError unless `group` is True (the default group) or a torch.distributed ProcessGroup this process belongs to,
    with torch.distributed initialised."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()):
        raise ValueError("process_group needs an initialised torch.distributed")
    if group is not True and not isinstance(group, dist.ProcessGroup):
        raise ValueError("process_group must be True (the default group) or a torch.distributed ProcessGroup, got %r" % (group,))
    if dist.get_rank(None if group is True else group) < 0:
        raise ValueError("this process is not a member of process_group")


def ranks_agree(refusal: Optional[str], config, group=True):
    """The agreement check of a collective call over the ranks of `group` (True: the default group): ONE
    all_gather_object of (this rank's refusal message or None, this rank's config as (field, value) pairs in a fixed
    order).  Every rank reads the same gathered list, so every rank raises the same ValueError -- naming the first rank
    that refused, or else the first rank and field that differ from group rank 0's -- or none does; no rank is left
    waiting in a later collective."""
    import torch.distributed as dist
    g = None if group is True else group
    got = [None] * dist.get_world_size(g)
    dist.all_gather_object(got, (refusal, tuple(config)), group=g)
    for r, (msg, _) in enumerate(got):
        if msg is not None:
            raise ValueError("rank %d refused: %s" % (r, msg))
    base = dict(got[0][1])
    for r, (_, cfg) in enumerate(got[1:], 1):
        for field, value in cfg:
            if value != base.get(field):
                raise ValueError("rank %d passed %s = %r, rank 0 %r" % (r, field, value, base.get(field)))


def check_td3_options(twin_critics, policy_delay, target_noise, target_noise_clip, group=None):
    """ValueError unless policy_delay >= 1, target_noise >= 0 and target_noise_clip >= 0.  Sharded (group not None): every
    rank checks its own arguments and ranks_agree compares the refusals and the four values, so every rank raises the
    same ValueError or none does -- a rank with another twin_critics or policy_delay would otherwise wait forever in a
    collective of a step the others do not run."""
    refusal = None
    if int(policy_delay) != policy_delay or policy_delay < 1:
        refusal = "policy_delay must be an integer >= 1, got %r" % (policy_delay,)
    elif not float(target_noise) >= 0.0:
        refusal = "target_noise must be >= 0, got %r" % (target_noise,)
    elif not float(target_noise_clip) >= 0.0:
        refusal = "target_noise_clip must be >= 0, got %r" % (target_noise_clip,)
    if group is None:
        if refusal is not None:
            raise ValueError(refusal)
        return
    check_process_group(group)
    ranks_agree(refusal, (("twin_critics", bool(twin_critics)), ("policy_delay", policy_delay), ("target_noise", float(target_noise)),
                          ("target_noise_clip", float(target_noise_clip))), group)


def _device_collective(t: torch.Tensor, g) -> bool:
    """True when a collective of group `g` takes `t` where it lies (a CUDA tensor and an NCCL backend); gloo takes a CPU copy."""
    import torch.distributed as dist
    return t.is_cuda and "nccl" in str(dist.get_backend(g))


def allreduce_counters(t: torch.Tensor, group=True) -> torch.Tensor:
    """The sum of an int64 counter tensor over the ranks of `group` (True: the default group) as a new CPU tensor; `t`
    itself is not changed.  One all-reduce: on the device for an NCCL group, on a CPU copy for gloo."""
    import torch.distributed as dist
    g = None if group is True else group
    s = t.clone() if _device_collective(t, g) else t.cpu().clone()
    dist.all_reduce(s, op=dist.ReduceOp.SUM, group=g)
    return s.cpu()


def _broadcast_rank0(t: torch.Tensor, group=True):
    """Overwrite `t` in place with group rank 0's `t` (on the device for an NCCL group, through a CPU copy for gloo)."""
    import torch.distributed as dist
    g = None if group is True else group
    if _device_collective(t, g):
        dist.broadcast(t, group=g, group_src=0)
    else:
        c = t.cpu()
        dist.broadcast(c, group=g, group_src=0)
        t.copy_(c)


class PeerExchange:
    """The gradient exchange of a sharded update over NVLink peer memory (csrc/ss_peer.cu): every rank
    owns an inbox {flags | 2 x world x capacity floats} shared with the other processes of the node
    through CUDA IPC; a rank's gradient reduction kernel stores its result into every inbox, and each
    rank's Adam kernel sums its inbox in rank order.  Replaces the NCCL all-reduce call between the
    gradient kernel and Adam (one node, up to 8 ranks)."""

    def __init__(self, group, device, capacity: int = max(A_N, C_N)):      # (ActorCritic passes its own sizes)
        import torch.distributed as dist
        g = None if group is True else group
        self.group, self.device, self.capacity = g, torch.device(device), int(capacity)
        self.world, self.rank = dist.get_world_size(g), dist.get_rank(g)
        if self.world > _lib.PEER_MAX_WORLD:
            raise ValueError("peer exchange supports up to %d ranks of one node" % _lib.PEER_MAX_WORLD)
        self._own = ctypes.c_void_p()
        self._imported = []
        with torch.cuda.device(self.device):
            check(lib.ss_peer_alloc(self.world, self.capacity, ctypes.byref(self._own)), "ss_peer_alloc")
            handle = (ctypes.c_ubyte * _lib.PEER_HANDLE_BYTES)()
            check(lib.ss_peer_export(self._own, handle), "ss_peer_export")
            handles = [None] * self.world
            dist.all_gather_object(handles, bytes(handle), group=g)
            self.bases = (ctypes.c_void_p * self.world)()
            for r, h in enumerate(handles):
                if r == self.rank:
                    self.bases[r] = self._own.value
                else:
                    buf = (ctypes.c_ubyte * _lib.PEER_HANDLE_BYTES).from_buffer_copy(h)
                    ptr = ctypes.c_void_p()
                    check(lib.ss_peer_import(buf, ctypes.byref(ptr)), "ss_peer_import")
                    self.bases[r] = ptr.value
                    self._imported.append(ptr)
        self.done_counter = torch.zeros(1, dtype=torch.int32, device=self.device)
        self.status = torch.zeros(1, dtype=torch.int32, device=self.device)
        self.epoch = 0
        dist.barrier(g)

    def reduce_push(self, workspace: torch.Tensor, parts: int, n_params: int, aux: Optional[torch.Tensor]):
        """Slices in `workspace` -> this rank's slot of every inbox; starts a new epoch."""
        self.epoch += 1
        with torch.cuda.device(self.device):
            check(lib.ss_peer_reduce_push(workspace.data_ptr(), int(parts), int(n_params), _ptr(aux), self.bases, self.world,
                                          self.rank, self.capacity, self.epoch, self.done_counter.data_ptr(),
                                          _stream(self.device)), "ss_peer_reduce_push")

    def check_status(self):
        if int(self.status.item()) & _lib.STATUS_PEER_TIMEOUT:
            self.status.zero_()
            raise RuntimeError("peer exchange: a rank's gradient never arrived")

    def close(self):
        with torch.cuda.device(self.device):
            torch.cuda.synchronize(self.device)
            for ptr in self._imported:
                lib.ss_peer_close(ptr)
            self._imported = []
            if self._own:
                import torch.distributed as dist
                if dist.is_initialized():
                    dist.barrier(self.group)          # nobody may still be storing into this inbox
                lib.ss_peer_free(self._own)
                self._own = ctypes.c_void_p()


class ActorCritic:
    """Actor and critic parameters, optimiser state and target copies on one GPU.

    Hyper-parameters default to the reference's: tf.keras Adam lr 1e-3, betas
    0.9 / 0.999, eps 1e-7 for both networks (SkillshotLearner.py:68, 118),
    Dropout(0.2) in the critic (SkillshotLearner.py:105).  gamma = 0 and tau = 1
    are the reference's update (critic regresses on the immediate reward, no
    target network); other values give DDPG proper.

    TD3 (no reference code, DESIGN.md section 6.14): twin_critics adds a second critic with its own slices of every
    buffer, [actor | pad | critic | pad | critic2], its own Adam step counter and its own initialisation (the critic's
    initialisers from a seed derived from `seed`).  One TD3 update (td3_step) computes
        y = r + gamma (1 - done) min(Q1'(s', a~), Q2'(s', a~)),  a~ = clamp(mu'(s') + clamp(target_noise eps, -c, c), -1, 1)
    with c = target_noise_clip (one critic without twin_critics; no draw when target_noise = 0), runs a critic step on
    critic 1 and then on critic 2 against that y, and on every policy_delay-th update only the actor step against
    critic 1.  The targets of all networks are soft-updated on those delayed updates only: the other updates pass tau = 0
    to the Adam kernels, and target = 0 w + 1 target leaves every target byte-identical.  The defaults (False, 1, 0, any
    clip) are the DDPG update of this class, with the same allocations and checkpoints.
    """

    def __init__(self, device="cuda", seed: int = 0, lr_actor: float = 1e-3, lr_critic: float = 1e-3,
                 gamma: float = 0.0, tau: float = 1.0, dropout: float = 0.2, process_group=None,
                 update_precision: str = "f32", collective: str = "nccl", frames: int = 1, twin_critics: bool = False,
                 policy_delay: int = 1, target_noise: float = 0.0, target_noise_clip: float = 0.5):
        check_td3_options(twin_critics, policy_delay, target_noise, target_noise_clip, process_group)
        self.twin_critics, self.policy_delay = bool(twin_critics), int(policy_delay)
        self.target_noise, self.target_noise_clip = float(target_noise), float(target_noise_clip)
        # any non-default option: the TD3 update (td3_step) instead of the DDPG one
        self.td3 = self.twin_critics or self.policy_delay > 1 or self.target_noise > 0.0
        if not torch.cuda.is_available():
            raise RuntimeError("skillshot_learning_b200 needs a CUDA device (no CPU fallback)")
        # frames > 1: the frame-stacked "planning" networks of readme.md:18-20 (no reference code): both first layers read
        # 12 * frames inputs, oldest frame first.  frames = 1 is the reference.  Their update runs on the exact float32
        # kernels (ss_*_frames) or, with update_precision "bf16", on the tensor cores (ss_*_frames_tc, separate steps).
        self.frames = int(frames)
        self.a_n, self.c_n = int(lib.ss_actor_frames_params(self.frames)), int(lib.ss_critic_frames_params(self.frames))
        if self.a_n < 0 or self.c_n < 0:
            raise ValueError("frames must be 1..20")
        self.actor_shapes = [(12 * self.frames, 256)] + ACTOR_SHAPES[1:]
        self.critic_shapes = [(12 * self.frames, 256)] + CRITIC_SHAPES[1:]
        self.device = torch.device(device)
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.seed = int(seed)
        self.lr_actor, self.lr_critic = float(lr_actor), float(lr_critic)
        self.beta1, self.beta2, self.eps = 0.9, 0.999, 1e-7
        self.gamma, self.tau, self.dropout = float(gamma), float(tau), float(dropout)
        self.group = process_group
        if update_precision not in ("f32", "bf16"):
            raise ValueError("update_precision must be 'f32' (exact path) or 'bf16' (tensor cores)")
        self.update_precision = update_precision     # gradient / TD-target kernels: float32 CUDA cores or tcgen05
        if collective not in ("nccl", "peer"):
            raise ValueError("collective must be 'nccl' (torch.distributed all-reduce) or 'peer' (fused NVLink exchange)")
        # the exchange step of a sharded update: an all-reduce call, or the fused peer-memory kernels
        self.peer = (PeerExchange(process_group, self.device, capacity=max(self.a_n, self.c_n))
                     if (process_group is not None and collective == "peer") else None)
        dev = self.device
        A_N, C_N = self.a_n, self.c_n
        # one allocation: [actor | pad | critic] so both vectors are 16-byte aligned (twin critics: [.. | pad | critic2])
        self._a_off, self._c_off = 0, (A_N + 3) // 4 * 4
        total = self._c_off + C_N
        if self.twin_critics:
            self._c2_off = (total + 3) // 4 * 4
            total = self._c2_off + C_N
        self.params = torch.zeros(total, dtype=torch.float32, device=dev)
        self.grads = torch.zeros(total, dtype=torch.float32, device=dev)
        self.adam_m = torch.zeros(total, dtype=torch.float32, device=dev)
        self.adam_v = torch.zeros(total, dtype=torch.float32, device=dev)
        self.target = torch.zeros(total, dtype=torch.float32, device=dev)
        self.stats = torch.zeros(2, dtype=torch.float32, device=dev)        # [sum sq err, sum q] of the last steps
        # gradient slices: one per CTA of the gradient kernels (at most 160 of them run: 148 SMs, one CTA each for the wide nets)
        self._ws_base = (int(lib.ss_learner_workspace_bytes()) if self.frames == 1
                         else 160 * (max(A_N, C_N) + 1) * 4)
        self.workspace = torch.empty(self._ws_base, dtype=torch.uint8, device=dev)
        self.step_actor = 0
        self.step_critic = 0
        if self.twin_critics:
            self.step_critic2 = 0
            self.critic2_sse = torch.zeros(1, dtype=torch.float32, device=dev)    # critic 2's sum sq err of its last step
        self.td3_updates = 0        # TD3 updates so far: phases the delayed actor / target updates
        self.counter = 0            # Philox counter: advances with every noisy call
        self._update_args = None    # cached ss_ddpg_update argument block (pointers change rarely)
        self._pair_mail = None      # ss_actor_critic_forward_tc's mailbox, allocated with the argument block
        self.init_weights(seed)

    # -- parameter views -----------------------------------------------------
    @property
    def actor(self):
        return self.params[self._a_off:self._a_off + self.a_n]

    @property
    def critic(self):
        return self.params[self._c_off:self._c_off + self.c_n]

    @property
    def target_actor(self):
        return self.target[self._a_off:self._a_off + self.a_n]

    @property
    def target_critic(self):
        return self.target[self._c_off:self._c_off + self.c_n]

    @property
    def critic2(self):
        return self._slice(self.params, "critic2")

    @property
    def target_critic2(self):
        return self._slice(self.target, "critic2")

    def _slice(self, buf, which):
        if which == "actor":
            return buf[self._a_off:self._a_off + self.a_n]
        if which == "critic2":
            if not self.twin_critics:
                raise ValueError("critic2 exists with twin_critics=True only")
            return buf[self._c2_off:self._c2_off + self.c_n]
        return buf[self._c_off:self._c_off + self.c_n]

    def _critic_init(self, g):
        c = []
        for i, s in enumerate(self.critic_shapes):
            if len(s) == 1:
                c.append(torch.zeros(s))
            elif i == 4:
                c.append(torch.randn(s, generator=g) * 0.05)
            else:
                lim = float(np.sqrt(6.0 / (s[0] + s[1])))
                c.append((torch.rand(s, generator=g) * 2.0 - 1.0) * lim)
        return torch.cat([t.reshape(-1) for t in c])

    def init_weights(self, seed: int):
        """Keras initialisers of the reference's layers: actor kernels RandomNormal(0, 0.05)
        (SkillshotLearner.py:74), critic hidden kernels glorot-uniform (the Dense default),
        critic output kernel "RandomNormal" = N(0, 0.05) (SkillshotLearner.py:113), biases 0.
        Twin critics: critic 2 takes the critic's initialisers from its own generator, seeded with `seed` mixed by a
        64-bit odd constant, so that it differs from critic 1."""
        g = torch.Generator(device="cpu")
        g.manual_seed(int(seed))
        a = [torch.randn(s, generator=g) * 0.05 if len(s) == 2 else torch.zeros(s) for s in self.actor_shapes]
        c = self._critic_init(g)
        c2 = None
        if self.twin_critics:
            g2 = torch.Generator(device="cpu")
            g2.manual_seed((int(seed) * 0x9E3779B97F4A7C15 + 0x632BE59BD9B4E019) % (1 << 63))
            c2 = self._critic_init(g2)
        self.set_weights(torch.cat([t.reshape(-1) for t in a]), c, critic2=c2)

    def set_weights(self, actor=None, critic=None, reset_optimizer: bool = True, *, critic2=None):
        """Install flat parameter vectors (Keras get_weights() order); targets are set equal.  critic2: the second critic
        of twin critics (ValueError without them)."""
        if critic2 is not None and not self.twin_critics:
            raise ValueError("critic2 needs twin_critics=True")
        if actor is not None:
            self.actor.copy_(_f32(actor, self.device, (self.a_n,)))
        if critic is not None:
            self.critic.copy_(_f32(critic, self.device, (self.c_n,)))
        if critic2 is not None:
            self.critic2.copy_(_f32(critic2, self.device, (self.c_n,)))
        self.target.copy_(self.params)
        if reset_optimizer:
            self.adam_m.zero_()
            self.adam_v.zero_()
            self.step_actor = self.step_critic = 0
            if self.twin_critics:
                self.step_critic2 = 0

    def get_weights(self, which="actor"):
        """List of numpy arrays like keras Model.get_weights() ("actor", "critic" or, with twin critics, "critic2")."""
        flat = self._slice(self.params, which).detach().cpu().numpy()
        return [w.copy() for w in split_params(flat, self.actor_shapes if which == "actor" else self.critic_shapes)]

    # -- forward ---------------------------------------------------------------
    def actor_forward(self, obs, param_noise_sd: float = 0.0, noise_group: int = 1, action_noise_sd: float = 0.0,
                      out: Optional[torch.Tensor] = None, target: bool = False, counter: Optional[int] = None,
                      precision: str = "f32"):
        """actions [n,2] = actor(obs [n,12]) (model_act*, SkillshotLearner.py:215-281).  frames > 1: obs [n, 12 * frames],
        oldest frame first, float32 kernels, no noise (FrameStackActor is the acting path of the stacked networks)."""
        obs = _f32(obs, self.device).reshape(-1, 12 * self.frames)
        n = obs.shape[0]
        if out is None:
            out = torch.empty((n, 2), dtype=torch.float32, device=self.device)
        theta = self.target_actor if target else self.actor
        if self.frames > 1:
            if param_noise_sd > 0 or action_noise_sd > 0 or precision != "f32":
                raise ValueError("frame-stacked networks: plain float32 forward only (see FrameStackActor)")
            with torch.cuda.device(self.device):      # dense ordered rows = a history ring read from slot 0
                check(lib.ss_actor_forward_frames(theta.data_ptr(), 0, 0, obs.data_ptr(), self.frames, self.frames - 1,
                                                  out.data_ptr(), n, _stream(self.device)), "ss_actor_forward_frames")
            return out
        if counter is None:
            counter = self.counter
            if param_noise_sd > 0 or action_noise_sd > 0:
                self.counter += 1
        if precision not in ("f32", "bf16"):
            raise ValueError("precision must be 'f32' (exact path) or 'bf16' (tensor cores)")
        fn = lib.ss_actor_forward if precision == "f32" else lib.ss_actor_forward_tc
        with torch.cuda.device(self.device):
            check(fn(theta.data_ptr(), obs.data_ptr(), out.data_ptr(), n, float(param_noise_sd), int(noise_group),
                     float(action_noise_sd), self.seed, int(counter), _stream(self.device)), "ss_actor_forward")
        return out

    def noisy_actor_params(self, sd: float, group: int = 0, counter: Optional[int] = None):
        """The perturbed parameter vector actor_forward uses for one noise group."""
        out = torch.empty(self.a_n, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            check(lib.ss_param_noise(self.actor.data_ptr(), out.data_ptr(), self.a_n, float(sd), self.seed, int(group),
                                     int(self.counter if counter is None else counter), _stream(self.device)),
                  "ss_param_noise")
        return out

    def critic_forward(self, obs, act, target: bool = False, precision: str = "f32", want_dq_da: bool = False):
        """q [n] = critic([obs, act]) with Dropout off; with want_dq_da (bf16 path) also -dQ/da [n,2]."""
        obs, act = _f32(obs, self.device).reshape(-1, 12 * self.frames), _f32(act, self.device).reshape(-1, 2)
        n = obs.shape[0]
        q = torch.empty(n, dtype=torch.float32, device=self.device)
        phi = self.target_critic if target else self.critic
        with torch.cuda.device(self.device):
            if self.frames > 1 and precision == "bf16":
                up = torch.empty((n, 2), dtype=torch.float32, device=self.device) if want_dq_da else None
                ws = self._workspace_for(n, "bf16")
                check(lib.ss_critic_forward_frames_tc(phi.data_ptr(), self.frames, obs.data_ptr(), act.data_ptr(), q.data_ptr(),
                                                      _ptr(up), n, ws.data_ptr(), ws.numel(), _stream(self.device)),
                      "ss_critic_forward_frames_tc")
                return (q, up) if want_dq_da else q
            if self.frames > 1:
                if precision != "f32":
                    raise ValueError("precision must be 'f32' (exact path) or 'bf16' (tensor cores)")
                check(lib.ss_critic_forward_frames(phi.data_ptr(), self.frames, obs.data_ptr(), act.data_ptr(), q.data_ptr(), n,
                                                   _stream(self.device)), "ss_critic_forward_frames")
                return q
            if precision == "bf16":
                up = torch.empty((n, 2), dtype=torch.float32, device=self.device) if want_dq_da else None
                check(lib.ss_critic_forward_tc(phi.data_ptr(), obs.data_ptr(), act.data_ptr(), n, q.data_ptr(), _ptr(up),
                                               None, None, 0.0, None, _stream(self.device)), "ss_critic_forward_tc")
                return (q, up) if want_dq_da else q
            check(lib.ss_critic_forward(phi.data_ptr(), obs.data_ptr(), act.data_ptr(), q.data_ptr(), n,
                                        _stream(self.device)), "ss_critic_forward")
        return q

    def td_targets(self, reward, next_obs, done=None, row_offset: int = 0):
        """y = r + gamma (1 - done) Q'(s', mu'(s')); gamma = 0 returns the reward itself
        (the reference's critic target, SkillshotLearner.py:434).  With the TD3 options the target is the class
        docstring's (ss_td3_targets*): the smoothing draw is keyed by the global row (row_offset + i) and the Philox
        counter, which then advances; target_noise = 0 draws nothing."""
        reward = _f32(reward, self.device).reshape(-1)
        if self.gamma == 0.0:
            return reward
        next_obs = _f32(next_obs, self.device).reshape(-1, 12 * self.frames)
        y = torch.empty_like(reward)
        if done is not None:
            done = done.to(device=self.device, dtype=torch.uint8).contiguous()
        n = reward.shape[0]
        if self.td3:
            if self.update_precision == "bf16":
                ws = self._workspace_for(n)
                fn, args = ((lib.ss_td3_targets_frames_tc, (self.frames,)) if self.frames > 1 else (lib.ss_td3_targets_tc, ()))
            else:
                ws, fn, args = None, lib.ss_td3_targets_frames, (self.frames,)
            with torch.cuda.device(self.device):
                check(fn(self.target_actor.data_ptr(), self.target_critic.data_ptr(),
                         self.target_critic2.data_ptr() if self.twin_critics else None, *args, reward.data_ptr(),
                         next_obs.data_ptr(), _ptr(done), self.gamma, self.target_noise, self.target_noise_clip, self.seed,
                         self.counter, int(row_offset), y.data_ptr(), n, _ptr(ws), 0 if ws is None else ws.numel(),
                         _stream(self.device)), "ss_td3_targets")
            if self.target_noise > 0.0:
                self.counter += 1
            return y
        with torch.cuda.device(self.device):
            if self.update_precision == "bf16" and self.frames > 1:
                ws = self._workspace_for(n)
                check(lib.ss_ddpg_targets_frames_tc(self.target_actor.data_ptr(), self.target_critic.data_ptr(), self.frames,
                                                    reward.data_ptr(), next_obs.data_ptr(), _ptr(done), self.gamma, y.data_ptr(),
                                                    n, ws.data_ptr(), ws.numel(), _stream(self.device)), "ss_ddpg_targets_frames_tc")
            elif self.update_precision == "bf16":
                ws = self._workspace_for(n)
                check(lib.ss_ddpg_targets_tc(self.target_actor.data_ptr(), self.target_critic.data_ptr(),
                                             reward.data_ptr(), next_obs.data_ptr(), _ptr(done), self.gamma,
                                             y.data_ptr(), n, ws.data_ptr(), ws.numel(), _stream(self.device)),
                      "ss_ddpg_targets_tc")
            else:
                check(lib.ss_ddpg_targets_frames(self.target_actor.data_ptr(), self.target_critic.data_ptr(), self.frames,
                                                 reward.data_ptr(), next_obs.data_ptr(), _ptr(done), self.gamma, y.data_ptr(), n,
                                                 _stream(self.device)), "ss_ddpg_targets")
        return y

    def _workspace_for(self, n: int, precision: Optional[str] = None) -> torch.Tensor:
        """Scratch for the gradient kernels: per-CTA gradient slices (+ 32 bytes per row for the
        tensor-core entry points: actions, -dQ/da and Q of the actor step; frames > 1: the slices and the tiles passed
        between the kernels of a call, ss_learner_frames_tc_workspace_bytes)."""
        bf16 = (precision or self.update_precision) == "bf16"
        if bf16 and self.frames > 1:
            need = max(self._ws_base, int(lib.ss_learner_frames_tc_workspace_bytes(self.frames, n)))
        else:
            need = self._ws_base + (32 * n if bf16 else 0)
        if self.workspace.numel() < need:
            self.workspace = torch.empty(need, dtype=torch.uint8, device=self.device)
        return self.workspace

    # -- update ----------------------------------------------------------------
    def _allreduce(self, t):
        allreduce_sum(t, self.group)

    def _sse(self, which: str) -> torch.Tensor:
        """The device slot of a critic's sum of squared errors: stats[0] for critic 1, critic2_sse for critic 2."""
        return self.critic2_sse if which == "critic2" else self.stats[0:1]

    def critic_grad(self, obs, act, y, keep=None, n_global: int = 0, row_offset: int = 0, slices_only: bool = False,
                    which: str = "critic"):
        """grads[critic] <- d/dphi mean (q - y)^2 of this (shard of a) batch; returns the gradient view.
        slices_only: leave the per-CTA slices in the workspace and return their number (peer exchange).
        which: "critic", or "critic2" with twin critics (its own slices of params / grads, its sum in critic2_sse)."""
        obs, act = _f32(obs, self.device).reshape(-1, 12 * self.frames), _f32(act, self.device).reshape(-1, 2)
        y = _f32(y, self.device).reshape(-1)
        n = obs.shape[0]
        if keep is not None:
            keep = torch.as_tensor(keep).to(device=self.device, dtype=torch.uint8).contiguous()
        g = self._slice(self.grads, which)
        phi = self._slice(self.params, which)
        ws = self._workspace_for(n)
        tail = (_ptr(keep), self.dropout, self.seed, self.counter, n, int(n_global), int(row_offset),
                None if slices_only else g.data_ptr(), self._sse(which).data_ptr(), ws.data_ptr(), ws.numel(), _stream(self.device))
        with torch.cuda.device(self.device):
            if self.update_precision == "bf16" and self.frames > 1:
                rc = lib.ss_critic_grad_frames_tc(phi.data_ptr(), self.frames, obs.data_ptr(), act.data_ptr(), y.data_ptr(),
                                                  *tail)
            elif self.update_precision == "bf16":
                rc = lib.ss_critic_grad_tc(phi.data_ptr(), obs.data_ptr(), act.data_ptr(), y.data_ptr(), *tail)
            else:
                rc = lib.ss_critic_grad_frames(phi.data_ptr(), self.frames, obs.data_ptr(), act.data_ptr(), y.data_ptr(), *tail)
        self.counter += 1
        if slices_only and rc > 0:
            return rc
        check(rc, "ss_critic_grad")
        return g

    def actor_grad(self, obs, slices_only: bool = False):
        """grads[actor] <- -sum_batch dQ/da da/dtheta (model_actor_fit_step, SkillshotLearner.py:395-410)."""
        obs = _f32(obs, self.device).reshape(-1, 12 * self.frames)
        g = self._slice(self.grads, "actor")
        ws = self._workspace_for(obs.shape[0])
        tail = (obs.data_ptr(), obs.shape[0], None if slices_only else g.data_ptr(), self.stats[1:2].data_ptr(), ws.data_ptr(),
                ws.numel(), _stream(self.device))
        with torch.cuda.device(self.device):
            if self.update_precision == "bf16" and self.frames > 1:
                rc = lib.ss_actor_grad_frames_tc(self.actor.data_ptr(), self.critic.data_ptr(), self.frames, *tail)
            elif self.update_precision == "bf16":
                rc = lib.ss_actor_grad_tc(self.actor.data_ptr(), self.critic.data_ptr(), *tail)
            else:
                rc = lib.ss_actor_grad_frames(self.actor.data_ptr(), self.critic.data_ptr(), self.frames, *tail)
        if slices_only and rc > 0:
            return rc
        check(rc, "ss_actor_grad")
        return g

    def _next_step(self, which: str):
        """Advance the Adam step counter of network `which`; returns (step, learning rate)."""
        if which == "actor":
            self.step_actor += 1
            return self.step_actor, self.lr_actor
        if which == "critic2":
            self.step_critic2 += 1
            return self.step_critic2, self.lr_critic
        self.step_critic += 1
        return self.step_critic, self.lr_critic

    def apply_adam(self, which: str, grad_scale: float = 1.0, from_peers: bool = False, tau: Optional[float] = None):
        """tf.keras Adam.apply_gradients on one network (+ soft target update with self.tau, or `tau` when given).
        from_peers: the gradient is the rank-ordered sum of this rank's peer inbox (fused exchange)."""
        n = self.a_n if which == "actor" else self.c_n
        step, lr = self._next_step(which)
        tau = self.tau if tau is None else float(tau)
        if from_peers:
            px = self.peer
            with torch.cuda.device(self.device):
                check(lib.ss_peer_adam_tf(px.bases[px.rank], px.world, px.capacity, px.epoch,
                                          self._slice(self.params, which).data_ptr(), self._slice(self.adam_m, which).data_ptr(),
                                          self._slice(self.adam_v, which).data_ptr(), self._slice(self.target, which).data_ptr(),
                                          self._slice(self.grads, which).data_ptr(), n, step, lr, self.beta1, self.beta2,
                                          self.eps, tau, float(grad_scale), px.status.data_ptr(), _stream(self.device)),
                      "ss_peer_adam_tf")
            return
        with torch.cuda.device(self.device):
            check(lib.ss_adam_tf(self._slice(self.params, which).data_ptr(), self._slice(self.grads, which).data_ptr(),
                                 self._slice(self.adam_m, which).data_ptr(), self._slice(self.adam_v, which).data_ptr(),
                                 self._slice(self.target, which).data_ptr(), n, step, lr, self.beta1, self.beta2,
                                 self.eps, tau, float(grad_scale), _stream(self.device)), "ss_adam_tf")

    def reduce_adam(self, which: str, parts: int, aux: Optional[torch.Tensor], grad_scale: float = 1.0,
                    tau: Optional[float] = None):
        """Single GPU: fixed-order sum of the `parts` gradient slices in the workspace + Adam + soft update, one kernel."""
        n = self.a_n if which == "actor" else self.c_n
        step, lr = self._next_step(which)
        tau = self.tau if tau is None else float(tau)
        with torch.cuda.device(self.device):
            check(lib.ss_reduce_adam_tf(self.workspace.data_ptr(), int(parts), n, _ptr(aux), self._slice(self.grads, which).data_ptr(),
                                        self._slice(self.params, which).data_ptr(), self._slice(self.adam_m, which).data_ptr(),
                                        self._slice(self.adam_v, which).data_ptr(), self._slice(self.target, which).data_ptr(),
                                        step, lr, self.beta1, self.beta2, self.eps, tau, float(grad_scale),
                                        _stream(self.device)), "ss_reduce_adam_tf")

    def critic_step(self, obs, act, y, keep=None, which: str = "critic", tau: Optional[float] = None):
        """One batch of model_critic.fit (SkillshotLearner.py:434): gradient of the batch-mean
        squared error, summed over the ranks when sharded, then Adam.  Returns the (device) sum of squared errors.
        which: "critic" or "critic2" (twin critics); tau: the soft update's tau instead of self.tau (TD3: 0 between
        delayed updates)."""
        _, n_global, row_offset = shard_info(int(np.prod(y.shape)), self.group)
        sse = self._sse(which)
        if self.group is not None and self.peer is None:      # NCCL: gradient -> all-reduce -> Adam
            g = self.critic_grad(obs, act, y, keep, n_global=n_global, row_offset=row_offset, which=which)
            self._allreduce(g)
            self.apply_adam(which, tau=tau)
            return sse[0]
        # per-CTA slices -> one kernel that sums them and applies Adam (single GPU), or pushes the sum into every
        # rank's inbox for the peers' Adam kernel (fused exchange)
        parts = self.critic_grad(obs, act, y, keep, n_global=n_global, row_offset=row_offset, slices_only=True, which=which)
        if self.peer is not None:
            self.peer.reduce_push(self.workspace, parts, self.c_n, sse)
            self.apply_adam(which, from_peers=True, tau=tau)
        else:
            self.reduce_adam(which, parts, sse, tau=tau)
        return sse[0]

    def actor_step(self, obs, tau: Optional[float] = None):
        """model_actor_fit_step (SkillshotLearner.py:386-417).  Returns the (device) sum of q."""
        if self.group is not None and self.peer is None:
            g = self.actor_grad(obs)
            self._allreduce(g)
            self.apply_adam("actor", tau=tau)
            return self.stats[1]
        parts = self.actor_grad(obs, slices_only=True)
        if self.peer is not None:
            self.peer.reduce_push(self.workspace, parts, self.a_n, self.stats[1:2])
            self.apply_adam("actor", from_peers=True, tau=tau)
        else:
            self.reduce_adam("actor", parts, self.stats[1:2], tau=tau)
        return self.stats[1]

    def td3_step(self, obs, act, reward, next_obs, done=None):
        """One TD3 update on a (shard of a) minibatch (class docstring): the target, a critic step on critic 1 and one on
        critic 2 against the same y (each with its own Philox dropout draw: the counter advances per call), and on every
        policy_delay-th update the actor step against critic 1.  Only those delayed updates soft-update the targets; the
        others pass tau = 0, which leaves every target byte-identical.  Returns (critic 1's sum of squared errors, the
        sum of q of the last actor step), device scalars; critic 2's sum is in critic2_sse."""
        _, _, row_offset = shard_info(int(np.prod(reward.shape)), self.group)
        y = self.td_targets(reward, next_obs, done, row_offset=row_offset)
        delayed = (self.td3_updates + 1) % self.policy_delay == 0
        tau = self.tau if delayed else 0.0
        sse = self.critic_step(obs, act, y, tau=tau)
        if self.twin_critics:
            self.critic_step(obs, act, y, which="critic2", tau=tau)
        if delayed:
            self.actor_step(obs, tau=tau)
        self.td3_updates += 1
        return sse, self.stats[1]

    def update_from_ring(self, ring: "ReplayRing", batch: int, out: Optional[dict] = None, sample_early: bool = False):
        """One whole update step from ONE library call (ss_ddpg_update): sample `batch` rows of `ring`,
        TD target, critic step, actor step -- the launches critic_step / actor_step make, without the
        interpreter time between them.  Single GPU or the fused peer exchange (an NCCL all-reduce needs
        the host between the gradient and Adam: use the separate steps).  Returns the minibatch dict.
        sample_early: the caller guarantees that the previous launch on the stream neither writes the ring nor touches
        `out` (ss_ddpg_update_args.sample_early): the minibatch is gathered while that launch still runs."""
        if self.group is not None and self.peer is None:
            raise ValueError("update_from_ring needs collective='peer' when the update is sharded")
        if self.frames > 1:
            raise ValueError("the single-call update is built for the reference's 12-input networks: use the separate steps")
        if ring.size == 0:
            raise ValueError("sampling from an empty ring")
        dev = self.device
        if out is None or out["reward"].shape[0] != batch or "y" not in out:
            out = dict(obs=torch.empty((batch, 12), dtype=torch.float32, device=dev),
                       act=torch.empty((batch, 2), dtype=torch.float32, device=dev),
                       reward=torch.empty(batch, dtype=torch.float32, device=dev),
                       next_obs=torch.empty((batch, 12), dtype=torch.float32, device=dev),
                       done=torch.empty(batch, dtype=torch.uint8, device=dev),
                       indices=torch.empty(batch, dtype=torch.int64, device=dev),
                       y=torch.empty(batch, dtype=torch.float32, device=dev))
        _, n_global, row_offset = shard_info(batch, self.group)
        ws = self._workspace_for(batch)
        key = (ring.obs.data_ptr(), ring.next_obs.data_ptr(), ring.capacity, out["obs"].data_ptr(), out["y"].data_ptr(), ws.data_ptr(),
               ws.numel(), batch, id(self.peer))
        if self._update_args is None:
            self._update_args = {}
        a = self._update_args.get(key)      # one cached argument block per set of minibatch buffers (callers alternate two)
        if a is None:
            if len(self._update_args) >= 4:
                self._update_args.clear()
            a = self._update_args[key] = _lib.DdpgUpdateArgs()
            a.ring_obs, a.ring_act, a.ring_reward = ring.obs.data_ptr(), ring.act.data_ptr(), ring.reward.data_ptr()
            a.ring_next_obs, a.ring_done, a.capacity = ring.next_obs.data_ptr(), ring.done.data_ptr(), ring.capacity
            a.batch = batch
            for k in ("obs", "act", "reward", "next_obs", "done", "indices", "y"):
                setattr(a, k, out[k].data_ptr())
            for k in ("actor", "critic"):
                setattr(a, k, self._slice(self.params, k).data_ptr())
                setattr(a, "target_" + k, self._slice(self.target, k).data_ptr())
                setattr(a, "m_" + k, self._slice(self.adam_m, k).data_ptr())
                setattr(a, "v_" + k, self._slice(self.adam_v, k).data_ptr())
                setattr(a, "grad_" + k, self._slice(self.grads, k).data_ptr())
            a.stats = self.stats.data_ptr()
            a.workspace, a.workspace_bytes = ws.data_ptr(), ws.numel()
            # the actor -> critic forward pairs (TD target, actor step) as one launch each (ss_actor_critic_forward_tc), for
            # minibatches small enough that a forward launch is mostly set-up and pipeline fill; the mailbox is filled with its
            # empty mark here once and left so by every call (SS_UPDATE_PAIR=0: two launches each, for A/B measurements)
            # (measured, profiles/r2_update_pair_ab.txt: 162.5 -> 158.9 us at 65,536 rows, 236 -> 252 us at 131,072)
            if batch <= 65536 and os.environ.get("SS_UPDATE_PAIR", "1") != "0":
                if self._pair_mail is None or self._pair_mail.shape[0] != batch:
                    self._pair_mail = torch.full((batch, 2), _lib.PAIR_MAIL_EMPTY, dtype=torch.int32, device=dev)
                a.pair_mail = self._pair_mail.data_ptr()
            else:
                self._pair_mail = None
            if self.peer is not None:
                px = self.peer
                a.world, a.rank, a.peer_capacity = px.world, px.rank, px.capacity
                a.peer_bases = ctypes.cast(px.bases, ctypes.c_void_p)
                a.done_counter, a.status = px.done_counter.data_ptr(), px.status.data_ptr()
        a.size, a.replay_seed, a.replay_counter = ring.size, ring.seed, ring.counter
        a.gamma, a.tau, a.lr_actor, a.lr_critic = self.gamma, self.tau, self.lr_actor, self.lr_critic
        a.beta1, a.beta2, a.eps, a.dropout_rate = self.beta1, self.beta2, self.eps, self.dropout
        a.seed, a.counter = self.seed, self.counter
        a.step_critic, a.step_actor = self.step_critic + 1, self.step_actor + 1
        a.n_global, a.row_offset = n_global, row_offset
        a.tensor_cores = 1 if self.update_precision == "bf16" else 0
        a.sample_early = 1 if sample_early else 0
        if self.peer is not None:
            a.epoch = self.peer.epoch + 1
        with torch.cuda.device(dev):
            check(lib.ss_ddpg_update(ctypes.byref(a), _stream(dev)), "ss_ddpg_update")
        ring.counter += 1
        self.counter += 1
        self.step_critic += 1
        self.step_actor += 1
        if self.peer is not None:
            self.peer.epoch += 2
        return out

    # -- checkpoint ------------------------------------------------------------
    def state_dict(self):
        sd = dict(params=self.params.cpu(), target=self.target.cpu(), adam_m=self.adam_m.cpu(),
                  adam_v=self.adam_v.cpu(), step_actor=self.step_actor, step_critic=self.step_critic,
                  counter=self.counter, seed=self.seed)
        if self.td3:            # (the flat buffers above already hold critic 2's slices)
            sd["td3_updates"] = self.td3_updates
        if self.twin_critics:
            sd["step_critic2"] = self.step_critic2
        return sd

    def check_state_dict(self, sd):
        """ValueError for a checkpoint of one critic into a twin-critic learner, of twin critics into a one-critic
        learner, or of another parameter layout."""
        twin = "step_critic2" in sd
        if twin != self.twin_critics:
            raise ValueError("a checkpoint of %s does not load into a learner with %s"
                             % (("twin critics", "one critic") if twin else ("one critic", "twin critics")))
        if sd["params"].numel() != self.params.numel():
            raise ValueError("checkpoint parameter layout of %d floats, this learner's %d" % (sd["params"].numel(), self.params.numel()))

    def load_state_dict(self, sd):
        """check_state_dict's refusals come before anything is copied."""
        self.check_state_dict(sd)
        twin = "step_critic2" in sd
        if twin:
            self.step_critic2 = int(sd["step_critic2"])
        self.td3_updates = int(sd.get("td3_updates", 0))
        for k in ("params", "target", "adam_m", "adam_v"):
            getattr(self, k).copy_(sd[k].to(self.device))
        self.step_actor, self.step_critic = int(sd["step_actor"]), int(sd["step_critic"])
        self.counter, self.seed = int(sd["counter"]), int(sd["seed"])


class ReplayRing:
    """Device-resident replay ring (structure of arrays).  The reference keeps one episode in
    Python lists and uses it once (SkillshotLearner.py:292-361); a ring sized to the episode and
    read back in order is that buffer."""

    def __init__(self, capacity: int, device="cuda", seed: int = 0, frames: int = 1):
        self.capacity, self.device, self.seed = int(capacity), torch.device(device), int(seed)
        self.frames = int(frames)          # observation rows of 12 * frames floats (the frame-stacked networks' inputs)
        self.width = 12 * self.frames
        c, dev = self.capacity, self.device
        self.obs = torch.zeros((c, self.width), dtype=torch.float32, device=dev)
        self.act = torch.zeros((c, 2), dtype=torch.float32, device=dev)
        self.reward = torch.zeros(c, dtype=torch.float32, device=dev)
        self.next_obs = torch.zeros((c, self.width), dtype=torch.float32, device=dev)
        self.done = torch.zeros(c, dtype=torch.uint8, device=dev)
        self.pos = 0
        self.size = 0
        self.counter = 0

    def push(self, obs, act, reward, next_obs, done=None, done_div: int = 1):
        obs, next_obs = _f32(obs, self.device).reshape(-1, self.width), _f32(next_obs, self.device).reshape(-1, self.width)
        act, reward = _f32(act, self.device).reshape(-1, 2), _f32(reward, self.device).reshape(-1)
        n = obs.shape[0]
        if n > self.capacity:
            raise ValueError("push of %d rows into a ring of %d" % (n, self.capacity))
        if done is not None:
            done = done.to(device=self.device, dtype=torch.uint8).contiguous()
        with torch.cuda.device(self.device):
            check(lib.ss_replay_push_frames(self.obs.data_ptr(), self.act.data_ptr(), self.reward.data_ptr(),
                                            self.next_obs.data_ptr(), self.done.data_ptr(), self.capacity, self.pos, self.frames,
                                            obs.data_ptr(), act.data_ptr(), reward.data_ptr(), next_obs.data_ptr(),
                                            _ptr(done), int(done_div), n, _stream(self.device)), "ss_replay_push")
        self.pos = (self.pos + n) % self.capacity
        self.size = min(self.capacity, self.size + n)

    def state_dict(self):
        return dict(capacity=self.capacity, seed=self.seed, pos=self.pos, size=self.size, counter=self.counter, frames=self.frames,
                    **{k: getattr(self, k).cpu() for k in ("obs", "act", "reward", "next_obs", "done")})

    def load_state_dict(self, sd):
        if int(sd["capacity"]) != self.capacity:
            raise ValueError("checkpoint ring holds %d rows, this ring %d" % (sd["capacity"], self.capacity))
        for k in ("obs", "act", "reward", "next_obs", "done"):
            getattr(self, k).copy_(sd[k].to(self.device))
        self.seed, self.pos, self.size, self.counter = int(sd["seed"]), int(sd["pos"]), int(sd["size"]), int(sd["counter"])

    def sample(self, batch: int, indices=None, out: Optional[dict] = None):
        """dict(obs, act, reward, next_obs, done, indices) of `batch` rows: the rows `indices` or a
        uniform draw with replacement from the filled part of the ring."""
        if self.size == 0:
            raise ValueError("sampling from an empty ring")
        dev = self.device
        if out is None or out["reward"].shape[0] != batch:
            out = dict(obs=torch.empty((batch, self.width), dtype=torch.float32, device=dev),
                       act=torch.empty((batch, 2), dtype=torch.float32, device=dev),
                       reward=torch.empty(batch, dtype=torch.float32, device=dev),
                       next_obs=torch.empty((batch, self.width), dtype=torch.float32, device=dev),
                       done=torch.empty(batch, dtype=torch.uint8, device=dev),
                       indices=torch.empty(batch, dtype=torch.int64, device=dev))
        if indices is not None:
            indices = torch.as_tensor(indices).to(device=dev, dtype=torch.int64).contiguous()
            if indices.numel() != batch:
                raise ValueError("indices must have `batch` entries")
        with torch.cuda.device(dev):
            check(lib.ss_replay_sample_frames(self.obs.data_ptr(), self.act.data_ptr(), self.reward.data_ptr(),
                                       self.next_obs.data_ptr(), self.done.data_ptr(), self.capacity, self.size, self.frames,
                                       _ptr(indices), self.seed, self.counter, batch, out["obs"].data_ptr(),
                                       out["act"].data_ptr(), out["reward"].data_ptr(), out["next_obs"].data_ptr(),
                                       out["done"].data_ptr(), out["indices"].data_ptr(), _stream(dev)),
                  "ss_replay_sample")
        self.counter += 1
        return out


class SkillshotLearner:
    """The reference SkillshotLearner surface (SkillshotLearner.py:12-693) over the CUDA
    library: one SkillshotGame, two players sharing one actor, critic fitted on the
    immediate reward, actor stepped along dQ/da, multiplicative parameter noise.

    Hyper-parameters are plain attributes as in the reference
    (`learner.model_param_game_tick_limit = 200`, SkillshotLearner.py:688).
    """
    game_state_features = list(FEATURE_KEYS)          # SkillshotLearner.py:17-36

    def __init__(self, device="cuda", seed: Optional[int] = None):
        seed = int(np.random.randint(0, 2 ** 31 - 1)) if seed is None else int(seed)
        # environment (SkillshotLearner.py:41-44)
        self.game_environment = SkillshotGame(device=device)
        self.player_ids = (1, 2)
        self.max_dist_normaliser = (2 * (250 ** 2)) ** 0.5
        self.use_random_start = True
        # dir locations (SkillshotLearner.py:47-51)
        self.save_location = "training_models"
        self.actor_dir_name = "actor"
        self.critic_dir_name = "critic"
        self.training_progress_dir_name = "training_progress"
        self.training_boards_dir_name = "training_boards"
        # model (SkillshotLearner.py:54-58)
        self.dim_state_space = 12
        self.dim_action_space = 2
        self.dim_reward_space = 1
        self.networks = ActorCritic(device=device, seed=seed)
        # model hyper-params (SkillshotLearner.py:61-64)
        self.model_param_batch_size = 16
        self.model_param_game_tick_limit = 2000
        self.action_noise_sd = 0.15
        self.param_noise_sd = 0.5
        self._rng = np.random.RandomState(seed)      # the shuffles the reference takes from np.random
        self.last_fit = {}

    # -- acting (SkillshotLearner.py:206-281) ------------------------------------
    def do_actions(self, player_id, predictions):
        player = self.game_environment.get_player_by_id(player_id)
        player.move_direction_float(float(predictions[0]))
        player.move_look_float(float(predictions[1]))
        player.move_shoot_projectile()           # attempted every time, SkillshotLearner.py:212-213

    def _predict(self, game_state, player_id, **noise):
        features = np.asarray(self.prepare_states([game_state], player_id)[0], dtype=np.float32)
        return self.networks.actor_forward(features[None, :], **noise).cpu().numpy()

    def model_act(self, game_state, player_id):
        predictions = self._predict(game_state, player_id)
        self.do_actions(player_id, predictions[0])
        return predictions

    def model_act_action_noise(self, game_state, player_id):
        predictions = self._predict(game_state, player_id, action_noise_sd=self.action_noise_sd)
        self.do_actions(player_id, predictions[0])
        return predictions

    def model_act_param_noise(self, game_state, player_id):
        predictions = self._predict(game_state, player_id, param_noise_sd=self.param_noise_sd, noise_group=1)
        self.do_actions(player_id, predictions[0])
        return predictions

    # -- dataset preparation (SkillshotLearner.py:512-573) ------------------------
    def prepare_states(self, game_states, player_id):
        board = self.game_environment.board_size
        cooldown_max = self.game_environment.get_player_by_id(player_id).projectile.cooldown_max
        norm = self.max_dist_normaliser
        rows = []
        for state in game_states:
            p = state.get(player_id)
            rows.append([
                p.get("player_path_dist_opponent") / norm,
                p.get("player_dist_opponent") / norm,
                p.get("player_pos_x") / board[0],
                p.get("player_pos_y") / board[1],
                (p.get("player_rotation") % 2 * np.pi) / 2 * np.pi,        # precedence as written, :529
                p.get("projectile_cooldown") / cooldown_max,
                p.get("projectile_dist_opponent") / norm,
                p.get("projectile_pos_x") / board[0],
                p.get("projectile_pos_y") / board[1],
                (p.get("projectile_rotation") % 2 * np.pi) / 2 * np.pi,
                p.get("projectile_path_dist_opponent") / norm,
                int(p.get("projectile_future_collision_opponent")),
            ])
        return rows

    @staticmethod
    def prepare_actions(actions, player_id):
        return [a[0] for a in actions.get(player_id)]

    @staticmethod
    def prepare_rewards(rewards, player_id):
        return list(rewards.get(player_id))

    # -- rewards (SkillshotLearner.py:575-603) -------------------------------------
    def calculate_rewards_looking(self, game_states):
        size = self.game_environment.board_size[0]
        return [{pid: -s[pid]["player_path_dist_opponent"] / size for pid in self.player_ids} for s in game_states]

    def calculate_rewards_simple(self, game_states):
        out = []
        for s in game_states:
            out.append({pid: s[pid]["projectile_dist_opponent"] - s[opp]["projectile_dist_opponent"]
                        for pid, opp in zip(self.player_ids, self.player_ids[::-1])})
        return out

    def calculate_rewards(self, game_states, on_target_multiplier_reduction=0.25, loss_reward_multiplier=2,
                          base_reward_multiplier=0.75):
        """The distance-shaped reward of SkillshotLearner.py:605-661, behaviour kept as written:
        reward = (opponent projectile's distance to me - multiplier * my projectile's distance to the
        opponent) / max_dist, multiplier 0.75, 0.5 while my projectile is on target, 2.75 for the player
        that was not `game_winner`; the `game_winner` player's entry at its projectile's firing tick is
        overwritten with 1.  The reference reads "projectile_cooldown" / "projectile_age" from the
        OUTER state dict where they do not exist, so its best-distance bonus is always 0 (:643-648)."""
        p1, p2 = self.player_ids
        rewards = []
        for index, state in enumerate(game_states):
            dist = {p1: state[p1]["projectile_dist_opponent"], p2: state[p2]["projectile_dist_opponent"]}
            loser_id = 0
            winner_id = state.get("game_winner")
            if winner_id != 0:
                rewards[index - state[winner_id]["projectile_age"]][winner_id] = 1    # Python indexing, as written
                loser_id = p2 if winner_id == p1 else p1
            entry = {}
            for pid, opp in ((p1, p2), (p2, p1)):
                multi = base_reward_multiplier
                if state[pid]["projectile_future_collision_opponent"]:
                    multi = base_reward_multiplier - on_target_multiplier_reduction
                if pid == loser_id:
                    multi = base_reward_multiplier + loss_reward_multiplier
                entry[pid] = ((dist[opp] - dist[pid] * multi) + 0 * 2) / self.max_dist_normaliser
            rewards.append(entry)
        return rewards

    # -- fitting (SkillshotLearner.py:386-443) --------------------------------------
    def model_actor_fit_step(self, state_tensor):
        """One deterministic-policy-gradient step of the actor on a batch of states."""
        self.networks.actor_step(np.asarray(state_tensor, dtype=np.float32))

    def models_fit(self, states, actions, rewards):
        assert len(states) == len(actions) == len(rewards)
        states = np.asarray(states, np.float32)
        actions = np.asarray(actions, np.float32).reshape(len(states), -1)
        rewards = np.asarray(rewards, np.float32)
        assert states.shape[0] == actions.shape[0] == rewards.shape[0]
        indices = np.arange(states.shape[0])
        self._rng.shuffle(indices)                                   # SkillshotLearner.py:426-431
        dev = self.networks.device
        s, a, r = (torch.from_numpy(x[indices]).to(dev) for x in (states, actions, rewards))
        bs = self.model_param_batch_size
        # critic.fit: one epoch, Keras reshuffles, batches of 16 with the short last batch kept
        order = torch.from_numpy(self._rng.permutation(len(indices))).to(dev)
        sse = torch.zeros((), device=dev)
        for b in range(0, len(indices), bs):
            idx = order[b:b + bs]
            sse += self.networks.critic_step(s[idx], a[idx], r[idx])
        # then the actor, consecutive batches of the shuffled states (SkillshotLearner.py:440-443)
        qsum = torch.zeros((), device=dev)
        for b in range(0, len(indices), bs):
            qsum += self.networks.actor_step(s[b:b + bs])
        self.last_fit = dict(critic_loss=float(sse) / len(indices), mean_q=float(qsum) / len(indices))

    # -- training loop (SkillshotLearner.py:283-384) -----------------------------------
    def model_train(self, epochs, save_progress=False, save_boards=False):
        total = dict(epoch_ticks=[], epoch_winner=[], epoch_board_sequences=[])
        game = self.game_environment
        for epoch in range(epochs):
            game.game_reset(random_positions=self.use_random_start)
            states, boards = [game.get_state()], []
            actions = {pid: [] for pid in self.player_ids}
            while game.game_live and game.ticks < self.model_param_game_tick_limit:
                game_state = states[-1]
                for pid in self.player_ids:      # both act from the same pre-tick state
                    actions[pid].append(self.model_act_param_noise(game_state, pid))
                game.game_tick()
                states.append(game.get_state())
                if save_boards:
                    boards.append(game.get_board())
            print("Begin Fitting for Epoch:", epoch)
            rewards_per_state = self.calculate_rewards_looking(states[1:])   # reward of action t = state t+1
            rewards = {pid: [r[pid] for r in rewards_per_state] for pid in self.player_ids}
            ts, ta, tr = [], [], []
            for pid in self.player_ids:                                      # P1 rows then P2 rows
                ts += self.prepare_states(states[:-1], pid)
                ta += self.prepare_actions(actions, pid)
                tr += self.prepare_rewards(rewards, pid)
            ts, ta, tr = np.array(ts), np.array(ta), np.array(tr)
            assert ts.shape == ((len(states) - 1) * 2, self.dim_state_space)
            assert ta.shape == (ts.shape[0], self.dim_action_space) and tr.shape == (ts.shape[0],)
            self.models_fit(ts, ta, tr)
            total["epoch_ticks"].append(game.ticks)
            total["epoch_winner"].append(game.winner_id)
            if save_boards:
                total["epoch_board_sequences"].append(boards)
            print("Epoch {} Completed, ticks taken: {}, game winner: {}".format(epoch, game.ticks, game.winner_id))
        print("All Epochs Completed")
        if save_progress:                                    # SkillshotLearner.py:379-384
            self.save_actor_critic_models(epochs)
            self.save_training_progress(total)
        if save_boards:
            self.save_training_boards(total["epoch_board_sequences"])
        self.training_progress = total
        return total

    # -- persistence (SkillshotLearner.py:123-162, naming kept, bugs not) ------------------
    def save_actor_critic_models(self, epochs):
        """training_models/{actor,critic}/{start}_{end}_model.npz (the reference writes .h5 through
        Keras; same directory layout and epoch-range naming, arrays in get_weights() order), and next to them
        training_models/learner_state/{start}_{end}_state.pt: targets, Adam moments and step counters of THAT range."""
        name = None
        for which, dir_name in (("actor", self.actor_dir_name), ("critic", self.critic_dir_name)):
            d = os.path.join(self.save_location, dir_name)
            os.makedirs(d, exist_ok=True)
            ends = [int(f.split("_")[1]) for f in os.listdir(d) if f.endswith("_model.npz")]
            start = max(ends) + 1 if ends else 0                  # SkillshotLearner.py:153-157
            name = "%d_%d" % (start, start + epochs)
            np.savez(os.path.join(d, name + "_model.npz"), *self.networks.get_weights(which))
        d = os.path.join(self.save_location, "learner_state")
        os.makedirs(d, exist_ok=True)
        torch.save(self.networks.state_dict(), os.path.join(d, name + "_state.pt"))
        print("Actor and Critic Saved.")

    def save_training_progress(self, total_progress):
        """training_models/training_progress/training_progress.csv, appended (SkillshotLearner.py:164-173):
        one row per epoch with its tick count and winner (the board rasters go to save_training_boards)."""
        import pandas as pd
        d = os.path.join(self.save_location, self.training_progress_dir_name)
        os.makedirs(d, exist_ok=True)
        frame = pd.DataFrame(dict(epoch_ticks=total_progress["epoch_ticks"], epoch_winner=total_progress["epoch_winner"]))
        path = os.path.join(d, "training_progress.csv")
        frame.to_csv(path, mode="a", header=not os.path.exists(path))
        print("Training Progress Saved")

    def load_training_progress(self):
        import pandas as pd
        return pd.read_csv(os.path.join(self.save_location, self.training_progress_dir_name, "training_progress.csv"))

    def save_training_boards(self, epoch_board_list):
        """training_models/training_boards/training_boards.npy: per epoch the list of 250 x 250 rasters
        (SkillshotLearner.py:182-193), the input of SkillshotGameDisplay.display_sequence."""
        d = os.path.join(self.save_location, self.training_boards_dir_name)
        os.makedirs(d, exist_ok=True)
        arr = np.empty(len(epoch_board_list), dtype=object)          # epochs differ in length: ragged
        for k, boards in enumerate(epoch_board_list):
            arr[k] = np.asarray(boards)
        np.save(os.path.join(d, "training_boards"), arr, allow_pickle=True)
        print("Training Boards Saved")

    def load_training_boards(self):
        return np.load(os.path.join(self.save_location, self.training_boards_dir_name, "training_boards.npy"), allow_pickle=True)

    def load_actor_critic_models(self, load_index=-1):
        """Loads the `load_index`-th saved actor and critic (sorted by their end epoch, SkillshotLearner.py:123-137) and, when
        it exists, the optimiser state saved WITH THAT epoch range.  Returns True, or False when a directory holds no model
        (as the reference does; its assignment to a loop variable, which loaded nothing, is not reproduced)."""
        flat, names = {}, {}
        for which, dir_name in (("actor", self.actor_dir_name), ("critic", self.critic_dir_name)):
            d = os.path.join(self.save_location, dir_name)
            files = sorted((f for f in os.listdir(d) if f.endswith("_model.npz")), key=lambda x: int(x.split("_")[1])) if os.path.isdir(d) else []
            if len(files) == 0:
                print("Failed to load: ", d)
                return False
            try:
                chosen = files[load_index]
            except IndexError:
                print("Failed to load: ", d)
                return False
            z = np.load(os.path.join(d, chosen))
            flat[which] = np.concatenate([z[k].ravel() for k in z.files])
            names[which] = chosen[:-len("_model.npz")]
        self.networks.set_weights(flat["actor"], flat["critic"])
        state = os.path.join(self.save_location, "learner_state", names["actor"] + "_state.pt")
        if names["actor"] == names["critic"] and os.path.exists(state):
            sd = torch.load(state, map_location="cpu", weights_only=False)
            # the weights of the chosen files stay; the optimiser moments, targets and counters of the same range come back
            for k in ("target", "adam_m", "adam_v"):
                getattr(self.networks, k).copy_(sd[k].to(self.networks.device))
            self.networks.step_actor, self.networks.step_critic = int(sd["step_actor"]), int(sd["step_critic"])
            self.networks.counter = int(sd["counter"])
        return True


class FrameStackActor:
    """The "planning" actor of readme.md:18-20 (BASELINE.json configs[4]; no reference code, parity unpinned): the
    actor of model_define_actor with a first layer that reads the last `frames` observations of its player,
    12 * frames -> 256 relu -> 128 relu -> 2 tanh.  frames = 1 is the reference actor.  precision "f32": the exact
    float32 kernels; "bf16": the tensor-core kernels (ss_frames_tc.cu).  Exploration by parameter noise with one
    perturbed parameter vector per noise group.
    """

    def __init__(self, n_rows: int, frames: int = 20, device="cuda", seed: int = 0, precision: str = "f32",
                 params: Optional[torch.Tensor] = None, learner_stack: bool = False):
        """params: the actor's flat parameter vector to act with (e.g. ActorCritic(frames=...).actor, so that the learner's
        updates are what acts), default a fresh RandomNormal(0, 0.05) vector.  learner_stack: with the tensor-core path
        (whose history is fp16 operand tiles) also keep the float32 history the learner's dense input rows are cut from."""
        if precision not in ("f32", "bf16"):
            raise ValueError("precision must be 'f32' (exact path) or 'bf16' (tensor cores)")
        self.precision = precision
        self._ws = None
        if not torch.cuda.is_available():
            raise RuntimeError("skillshot_learning_b200 needs a CUDA device (no CPU fallback)")
        self.device = torch.device(device)
        self.n_rows, self.frames, self.seed = int(n_rows), int(frames), int(seed)
        self.n_params = int(lib.ss_actor_frames_params(self.frames))
        if self.n_params < 0 or self.frames > 20:
            raise ValueError("frames must be 1..20")
        g = torch.Generator(device="cpu").manual_seed(self.seed)
        shapes = [(12 * self.frames, 256), (256,), (256, 128), (128,), (128, 2), (2,)]
        parts = [torch.randn(sh, generator=g) * 0.05 if len(sh) == 2 else torch.zeros(sh) for sh in shapes]   # RandomNormal(0, 0.05)
        self.shapes = shapes
        if params is not None:
            if params.numel() != self.n_params or params.dtype != torch.float32 or not params.is_contiguous():
                raise ValueError("params must be a contiguous float32 vector of %d values" % self.n_params)
            self.params = params
        else:
            self.params = torch.cat([p.reshape(-1) for p in parts]).to(self.device)
        self.stack32 = None
        if precision == "bf16" and learner_stack:
            self.stack32 = torch.zeros((self.n_rows, self.frames, 12), dtype=torch.float32, device=self.device)
        self._ordered = None
        if precision == "bf16":
            # the tensor-core path keeps the history as fp16 tiles in the MMA operand layout (ss_obs_stack_push_tc)
            self.stack = torch.zeros(int(lib.ss_obs_stack_tc_bytes(self.n_rows, self.frames)), dtype=torch.uint8, device=self.device)
        else:
            self.stack = torch.zeros((self.n_rows, self.frames, 12), dtype=torch.float32, device=self.device)
        self.head = -1                 # slot of the newest frame = head % frames
        self.counter = 0
        self._noisy = None

    def push(self, obs, done=None, done_div: int = 2):
        """Append the newest observation [n_rows,12]; rows whose game restarted (done, one flag per done_div rows)
        are refilled with it.  The first push fills every slot."""
        obs = _f32(obs, self.device).reshape(self.n_rows, 12)
        first = self.head < 0
        self.head += 1
        if first:
            done, done_div = torch.ones(self.n_rows, dtype=torch.uint8, device=self.device), 1
        elif done is not None:
            done = done.to(device=self.device, dtype=torch.uint8).contiguous()
        fn = lib.ss_obs_stack_push_tc if self.precision == "bf16" else lib.ss_obs_stack_push
        with torch.cuda.device(self.device):
            check(fn(self.stack.data_ptr(), self.n_rows, self.frames, self.head, obs.data_ptr(), _ptr(done), int(done_div),
                     _stream(self.device)), "ss_obs_stack_push")
            if self.stack32 is not None:
                check(lib.ss_obs_stack_push(self.stack32.data_ptr(), self.n_rows, self.frames, self.head, obs.data_ptr(), _ptr(done),
                                            int(done_div), _stream(self.device)), "ss_obs_stack_push")

    def ordered_rows(self, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """The network input of every row as dense float32 rows [n_rows, 12 * frames], oldest frame first: what the learner
        of the stacked networks stores and trains on (ss_obs_stack_ordered)."""
        src = self.stack if self.precision == "f32" else self.stack32
        if src is None:
            raise ValueError("tensor-core history only: construct with learner_stack=True")
        if out is None:
            out = torch.empty((self.n_rows, 12 * self.frames), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            check(lib.ss_obs_stack_ordered(src.data_ptr(), self.n_rows, self.frames, self.head, out.data_ptr(), _stream(self.device)),
                  "ss_obs_stack_ordered")
        return out

    def forward(self, param_noise_sd: float = 0.0, noise_group: int = 0, out: Optional[torch.Tensor] = None):
        """actions [n_rows,2] from the current stack; param_noise_sd > 0: rows i share the perturbed parameters of
        noise group i // noise_group (fresh draw per call)."""
        if self.head < 0:
            raise ValueError("push an observation first")
        if out is None:
            out = torch.empty((self.n_rows, 2), dtype=torch.float32, device=self.device)
        params, stride = self.params, 0
        with torch.cuda.device(self.device):
            if param_noise_sd > 0:
                if noise_group <= 0:
                    raise ValueError("noise_group must be positive")
                n_groups = (self.n_rows + noise_group - 1) // noise_group
                stride = (self.n_params + 3) // 4 * 4
                if self._noisy is None or self._noisy.numel() < n_groups * stride:
                    self._noisy = torch.empty(n_groups * stride, dtype=torch.float32, device=self.device)
                check(lib.ss_param_noise_groups(self.params.data_ptr(), self._noisy.data_ptr(), self.n_params, n_groups, stride,
                                                float(param_noise_sd), self.seed, self.counter, _stream(self.device)),
                      "ss_param_noise_groups")
                self.counter += 1
                params = self._noisy
            if self.precision == "bf16":
                need = int(lib.ss_actor_frames_tc_workspace_bytes(self.n_rows, int(noise_group) if stride else 0))
                if self._ws is None or self._ws.numel() < need:
                    self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
                check(lib.ss_actor_forward_frames_tc(params.data_ptr(), stride, int(noise_group), self.stack.data_ptr(), self.frames,
                                                     self.head, out.data_ptr(), self.n_rows, self._ws.data_ptr(), self._ws.numel(),
                                                     _stream(self.device)), "ss_actor_forward_frames_tc")
            else:
                check(lib.ss_actor_forward_frames(params.data_ptr(), stride, int(noise_group), self.stack.data_ptr(), self.frames,
                                                  self.head, out.data_ptr(), self.n_rows, _stream(self.device)),
                      "ss_actor_forward_frames")
        return out

    def ordered_stack(self) -> torch.Tensor:
        """[n_rows, frames * 12] network input, oldest frame first (introspection / tests)."""
        order = [(self.head + 1 + f) % self.frames for f in range(self.frames)]
        stack = self.stack
        if self.precision == "bf16":      # [tile][K / 8][128][8] fp16 -> [row][slot][12]
            tiles = (self.n_rows + 127) // 128
            x = stack.view(torch.float16).view(tiles, -1, 128, 8).permute(0, 2, 1, 3).reshape(tiles * 128, -1)
            stack = x[:self.n_rows, :self.frames * 12].float().reshape(self.n_rows, self.frames, 12)
        return stack[:, order, :].reshape(self.n_rows, self.frames * 12)


POOL_STRIDE = (A_N + 3) // 4 * 4          # floats between two opponent vectors (16-byte aligned)


def check_pool_blocks(blocks, pool_envs: int, n_opponents: int) -> list:
    """The block table as a list of ints: one even size >= 2 per opponent, summing to pool_envs; else ValueError."""
    out = [int(b) for b in blocks]
    if len(out) != int(n_opponents) or any(b < 2 or b % 2 for b in out) or sum(out) != int(pool_envs):
        raise ValueError("pool blocks must be %d even sizes >= 2 summing to %d, got %s" % (int(n_opponents), int(pool_envs), out))
    return out


def pool_layout(n_envs: int, pool_envs: int, n_opponents: int, blocks=None) -> np.ndarray:
    """int64 [n_envs, 2]: the row of each (env, player) when the last pool_envs envs are played against n_opponents frozen
    actors (include/skillshot_b200.h, "training against a pool").  Rows [0, L) are the learner's, L = 2 S + M with
    S = n_envs - M; rows L + r are opponent row r.  Self-play env i keeps rows 2i + p; opponent k owns the b_k pool envs
    from S + B_k, B_k = b_0 + ... + b_{k-1}, the learner being player 1 in the first b_k / 2 of them.  blocks: the b_k
    (check_pool_blocks); None: M / K each."""
    n, M = int(n_envs), int(pool_envs)
    S = n - M
    rows = np.empty((n, 2), np.int64)
    rows[:S] = np.arange(2 * S).reshape(S, 2)
    if M:
        K = int(n_opponents)
        j = np.arange(M)
        if blocks is None:
            b = M // K
            lp = (j % b >= b // 2).astype(np.int64)          # the learner's player in pool env S + j
        else:
            sizes = np.array(check_pool_blocks(blocks, M, K), np.int64)
            starts = np.concatenate([[0], np.cumsum(sizes)])
            k = np.searchsorted(starts, j, side="right") - 1
            lp = (j - starts[k] >= sizes[k] // 2).astype(np.int64)
        L = 2 * S + M
        rows[S + j, lp] = 2 * S + j
        rows[S + j, 1 - lp] = L + j
    return rows


PFSP_WEIGHTINGS = ("hard", "variance", "uniform")


def pfsp_blocks(scores, pool_envs: int, weighting: str = "hard", p: float = 2.0, min_envs: int = 2) -> list:
    """Prioritized fictitious self-play: the pool envs per opponent from the learner's score against each (1 win, 0.5 draw,
    0 loss; None or NaN for an opponent without finished games counts as 0.5).  Every opponent gets min_envs (even, >= 2);
    the rest is split in units of 2 envs in proportion to the weights -- "hard" (1 - s)^p, where play goes to the opponents
    the learner still loses to, "variance" s (1 - s), where it goes to the even matches, or "uniform" -- by largest
    remainder, ties to the lower k.  All weights 0 gives the uniform split.  Returns a list of ints summing to pool_envs."""
    if weighting not in PFSP_WEIGHTINGS:
        raise ValueError("weighting must be one of %s, got %r" % (PFSP_WEIGHTINGS, weighting))
    s = np.array([0.5 if v is None or math.isnan(float(v)) else float(v) for v in scores], np.float64)
    K, M, m, p = len(s), int(pool_envs), int(min_envs), float(p)
    if not 1 <= K <= _lib.LEAGUE_MAX_POLICIES:
        raise ValueError("1..%d scores, got %d" % (_lib.LEAGUE_MAX_POLICIES, K))
    if ((s < 0) | (s > 1)).any():
        raise ValueError("scores must lie in [0, 1]")
    if m < 2 or m % 2 or M % 2 or M < K * m:
        raise ValueError("pool_envs (%d) must be even and at least %d opponents x min_envs (%d, even, >= 2)" % (M, K, m))
    if not math.isfinite(p) or p < 0:
        raise ValueError("p must be finite and >= 0, got %r" % p)
    w = (1.0 - s) ** p if weighting == "hard" else s * (1.0 - s) if weighting == "variance" else np.ones(K)
    if w.sum() <= 0:
        w = np.ones(K)
    units = (M - K * m) // 2
    quota = units * w / w.sum()
    share = np.floor(quota).astype(np.int64)
    order = sorted(range(K), key=lambda k: (-(quota[k] - share[k]), k))
    for k in order[:units - int(share.sum())]:
        share[k] += 1
    return [m + 2 * int(u) for u in share]


class SelfPlayTrainer:
    """Batched self-play: E games stepped together, both players driven by the shared actor
    with parameter-noise exploration, transitions kept in a device replay ring, critic and
    actor updated on sampled minibatches.  One rank per GPU; with a process group the only
    exchange is the all-reduce of the flat gradients (envs and replay shard naturally).
    """

    def __init__(self, n_envs: int, device="cuda", seed: int = 0, replay_capacity: Optional[int] = None,
                 batch_size: int = 4096, gamma: float = 0.0, tau: float = 1.0, param_noise_sd: float = 0.5,
                 noise_group: int = 128, reward_mode: str = "looking", tick_limit: int = 2000,
                 random_positions: bool = True, process_group=None, precision: str = "f32", collective: str = "nccl",
                 frames: int = 1, update_precision: Optional[str] = None, opponents=None, pool_envs: Optional[int] = None,
                 pool_blocks=None, twin_critics: bool = False, policy_delay: int = 1, target_noise: float = 0.0,
                 target_noise_clip: float = 0.5):
        """frames > 1: the frame-stacked "planning" networks (readme.md:18-20, BASELINE.json configs[4]): both players act
        from their last `frames` observations (FrameStackActor; `precision` selects its float32 or tensor-core kernels),
        the replay ring stores the stacked observations, and the critic / actor update of SkillshotLearner.py:386-443 runs
        on the 12 * frames-input networks in separate steps.
        update_precision: the kernels of that update, "f32" or "bf16"; None = `precision` when frames = 1, "f32" when
        frames > 1.
        opponents: train against a pool of frozen actors (flat vectors or six get_weights() arrays of any frame count,
        copied here, at most 64): the last pool_envs envs (default: half of them, rounded down to a multiple of
        2 * len(opponents)) are the learner against opponent k in block k of pool_envs / len(opponents) envs, seat-balanced
        (pool_layout).  The opponents act without noise and only the learner's transitions are stored; an opponent with
        more than one frame keeps a history of its rows.  See set_opponent / pool_progress.
        pool_blocks: the pool envs of each opponent (even sizes >= 2 summing to pool_envs, pool_layout) instead of
        pool_envs / len(opponents) each; see set_pool_blocks / rebalance_pool.
        process_group with opponents (a sharded pool, DESIGN.md section 6.13): one rank per GPU, every rank passing the same
        n_envs, pool_envs, number of opponents, frames, opponent frame counts, pool_blocks and collective, and its own seed.
        The pool is replicated: every rank plays all K opponents on its own pool_envs envs with the same blocks, so a
        rank's rollout is the single-GPU pool rollout of its envs and the update sums gradients over the ranks as for
        sharded self-play.  process_group must be True (the default group) or a ProcessGroup of an initialised
        torch.distributed, else ValueError.  Every rank then checks the pool rules and one all_gather_object compares the
        ranks' refusals and configurations: when any rank refused or one differs, every rank raises the same ValueError
        before anything is allocated.  The opponents are then broadcast from group rank 0.  Every pool method
        (set_opponent, set_pool_blocks, rebalance_pool, pool_progress) is collective: call it on every rank with the same
        arguments, as update().  save / load write and read each rank's own file.
        twin_critics, policy_delay, target_noise, target_noise_clip: the TD3 update of ActorCritic (DESIGN.md section 6.14),
        which update() then runs through update_stepwise; the defaults are the DDPG update.  Bad values raise ValueError
        before anything is allocated (sharded: on every rank, when any rank refused or passed other values)."""
        check_td3_options(twin_critics, policy_delay, target_noise, target_noise_clip, process_group)
        self.device = torch.device(device)
        self.frames = int(frames)
        self.opponents, self.pool_envs, self.pool_stats = None, 0, None
        if opponents is not None:
            if process_group is not None:
                check_process_group(process_group)

            def pool_rules():
                K = len(opponents)
                if reward_mode == "simple":
                    raise ValueError("training against a pool supports reward modes none / looking / terminal")
                if not 1 <= K <= _lib.LEAGUE_MAX_POLICIES:
                    raise ValueError("1..%d opponents, got %d" % (_lib.LEAGUE_MAX_POLICIES, K))
                M = (int(n_envs) // 2) // (2 * K) * (2 * K) if pool_envs is None else int(pool_envs)
                if not 0 <= M <= int(n_envs) or M % (2 * K):
                    raise ValueError("pool_envs must be a multiple of 2 * %d in [0, n_envs], got %d" % (K, M))
                if precision == "bf16" and float(param_noise_sd) > 0 and int(noise_group) % 128:
                    raise ValueError("with tensor cores and parameter noise the noise group must be a multiple of 128, got %d" % noise_group)
                vecs = [actor_vector(a) for a in opponents]
                # None: M / K envs per opponent, the step of ss_pool_rollout (no block table is passed)
                blocks = None if pool_blocks is None else check_pool_blocks(pool_blocks, M, K)
                L = 2 * int(n_envs) - M
                if replay_capacity is not None and (replay_capacity % L or replay_capacity < 2 * L):
                    raise ValueError("with a pool the replay capacity must be a multiple of the %d learner rows, at least two of them" % L)
                if self.device.type != "cuda":
                    raise ValueError("device must be a CUDA device")
                return vecs, M, blocks

            if process_group is None:
                opp_vecs, M, self._blocks = pool_rules()
            else:
                # sharded: every rank runs the rules, then one exchange makes every rank raise, or none
                refusal, config = None, ()
                try:
                    opp_vecs, M, self._blocks = pool_rules()
                    config = (("n_envs", int(n_envs)), ("pool_envs", M), ("opponents", len(opp_vecs)), ("frames", self.frames),
                              ("opponent frames", [f for _, f in opp_vecs]),
                              ("pool_blocks", self._blocks or [M // len(opp_vecs)] * len(opp_vecs)), ("collective", collective))
                except ValueError as e:
                    refusal = str(e)
                ranks_agree(refusal, config, process_group)
            self.opp_frames = [f for _, f in opp_vecs]
            self.pool_envs = M
        self.learner_rows = 2 * int(n_envs) - self.pool_envs       # rows of the learner's transitions per tick
        L = self.learner_rows
        self.envs = SkillshotEnvs(n_envs, device=device, random_positions=random_positions, seed=seed,
                                  reward_mode=reward_mode, tick_limit=tick_limit, auto_reset=True)
        self.envs.collect_episode_stats = True     # the reference's per-episode ticks / winner log, reduced on the device
        self.networks = ActorCritic(device=device, seed=seed if process_group is None else 0, gamma=gamma, tau=tau,
                                    process_group=process_group,
                                    update_precision=update_precision or (precision if self.frames == 1 else "f32"),
                                    collective=collective, frames=self.frames, twin_critics=twin_critics,
                                    policy_delay=policy_delay, target_noise=target_noise, target_noise_clip=target_noise_clip)
        self.networks.seed = seed          # exploration / dropout streams differ per rank, weights do not
        self.replay = ReplayRing(replay_capacity or L * 8, device=device, seed=seed, frames=self.frames)
        self.batch_size, self.param_noise_sd, self.noise_group = int(batch_size), float(param_noise_sd), int(noise_group)
        self.precision = precision
        self.update_precision = update_precision
        n = n_envs
        self.obs = self.envs.observe().contiguous()                       # [n,2,12] seen by the actor next
        self.prev_obs = torch.empty_like(self.obs)
        self.actions = torch.empty((n, 2, 2), dtype=torch.float32, device=self.device)
        if opponents is not None:
            K = len(opp_vecs)
            # one row per opponent, as wide as the largest vector (16-byte aligned; POOL_STRIDE when all have one frame)
            self.opponents = torch.zeros((K, max((v.size + 3) // 4 * 4 for v, _ in opp_vecs)), dtype=torch.float32, device=self.device)
            for k, (v, _) in enumerate(opp_vecs):
                self.opponents[k, :v.size] = torch.from_numpy(v).to(self.device)
            if process_group is not None:
                _broadcast_rank0(self.opponents, process_group)      # the same pool on every rank by construction
            self.pool_stats = torch.zeros((K, _lib.POOL_STATS), dtype=torch.int64, device=self.device)
            # rows [0, L) the learner's, [L, 2n) the opponents' (pool_layout): observations and actions
            rows = torch.from_numpy(pool_layout(n, self.pool_envs, len(self.opponents), self._blocks).reshape(-1)).to(self.device)
            self.obs = torch.empty((2 * n, 12), dtype=torch.float32, device=self.device)
            self.obs[rows] = self.envs.observe().reshape(-1, 12)
            self.prev_obs = None
            self.actions = torch.empty((2 * n, 2), dtype=torch.float32, device=self.device)
            self._pool_reward = torch.zeros(L, dtype=torch.float32, device=self.device)
            self._pool_ws = None
            # the histories of the opponents with frames > 1, b_k rows each, filled with the first observation (slot 0);
            # every history of the pool shares one slot counter
            self._pool_head = 0      # (see pool_head)
            self._alloc_opp_stacks(0)
        self.stack = None
        if self.frames > 1:
            # the acting network IS the learner's actor vector; the history lives in the FrameStackActor (its L rows)
            self.stack = FrameStackActor(L, frames=self.frames, device=device, seed=seed, precision=precision,
                                         params=self.networks.actor, learner_stack=True)
            self.stack.push(self.obs[:L] if self.opponents is not None else self.obs.reshape(-1, 12))
            self.rows = self.stack.ordered_rows()                         # [L, 12 frames]: the stacked observation now
            self.prev_rows = torch.empty_like(self.rows) if self.opponents is None else None
        self._batch = None
        self._batches = [None, None]        # update(): two sets of minibatch buffers used in turn
        self._ring_clean = False            # no rollout (nothing of this object's that writes the ring) since the last update
        self.ticks = 0
        self.updates = 0
        self.exchange_check_every = 256     # updates between looks at the peer exchange's status word
        self._tile_ready, self._stream2 = None, None      # overlapped rollout (rollout()): allocated on first use

    @property
    def pool_head(self) -> int:
        """The slot counter of the newest frame shared by every history of the pool: the learner's FrameStackActor's when it
        reads more than one frame, else the trainer's own (then only the opponents' histories use it)."""
        return self.stack.head if self.stack is not None else self._pool_head

    @property
    def pool_blocks(self) -> list:
        """The pool envs of each opponent (pool_layout's blocks).  Per-env speeds (envs.set_speeds) belong to the env, not
        to the block: each opponent plays at the speeds of the envs its block covers."""
        if self.opponents is None:
            raise ValueError("this trainer has no opponent pool")
        K = len(self.opponents)
        return list(self._blocks) if self._blocks is not None else [self.pool_envs // K] * K

    def _alloc_opp_stacks(self, head: int, fill: bool = True):
        """A history of b_k rows for each opponent with frames > 1, every slot filled with its rows' current observation
        (fill) or zero (to be loaded)."""
        L, bf16 = self.learner_rows, self.precision == "bf16"
        self.opp_stacks = [None] * len(self.opponents)
        start = 0
        for k, (f, b) in enumerate(zip(self.opp_frames, self.pool_blocks)):
            if f > 1 and b > 0:
                s = (torch.zeros(int(lib.ss_obs_stack_tc_bytes(b, f)), dtype=torch.uint8, device=self.device) if bf16 else
                     torch.zeros((b, f, 12), dtype=torch.float32, device=self.device))
                if fill:
                    fn = lib.ss_obs_stack_push_tc if bf16 else lib.ss_obs_stack_push
                    ones = torch.ones(b, dtype=torch.uint8, device=self.device)
                    with torch.cuda.device(self.device):
                        check(fn(s.data_ptr(), b, f, int(head), self.obs[L + start:].data_ptr(), ones.data_ptr(), 1, _stream(self.device)),
                              "ss_obs_stack_push")
                self.opp_stacks[k] = s
            start += b

    def set_pool_blocks(self, blocks):
        """Lay the pool out again with blocks[k] envs for opponent k (even, >= 2, summing to pool_envs), between rollouts.
        Every pool game restarts (ss_pool_restart, Philox counter envs.counter, which then advances by one tick): moving an
        env between blocks can flip the learner's seat, and an opponent's history is indexed by the env's offset in its
        block.  The self-play envs, rows and histories are untouched.  The last stored transition of a restarted game keeps
        its next observation and a 0 done flag, as a tick-limit ending does; nothing is counted in pool_stats or the
        episode statistics.  Sharded: collective; one all-gather checks that every rank passed the same valid table, and
        otherwise every rank raises ValueError and nothing restarts."""
        if self.opponents is None:
            raise ValueError("this trainer has no opponent pool")
        n, M, K, L = self.envs.n_envs, self.pool_envs, len(self.opponents), self.learner_rows
        group = self.networks.group
        if group is None:
            blocks = check_pool_blocks(blocks, M, K)
        else:
            refusal = None
            try:
                blocks = check_pool_blocks(blocks, M, K)
            except ValueError as e:
                refusal, blocks = str(e), None
            ranks_agree(refusal, (("pool_blocks", blocks),), group)
        envs = self.envs
        table = (ctypes.c_int64 * K)(*blocks)
        with torch.cuda.device(self.device):
            check(lib.ss_pool_restart(envs.state.data_ptr(), n, M, K, table,
                                      _lib.RESET_RANDOM if envs.random_positions else _lib.RESET_FIXED, envs.seed, envs.counter,
                                      self.obs.data_ptr(), self.obs[L:].data_ptr(), envs.status.data_ptr(), _stream(self.device)),
                  "ss_pool_restart")
            envs.counter += 1
            st = self.stack
            if st is not None:
                # the learner's pool rows restart their histories; the self-play rows push their newest observation again
                done = torch.zeros(n, dtype=torch.uint8, device=self.device)
                done[n - M:] = 1
                check(lib.ss_obs_stack_push_pool(st.stack.data_ptr() if st.precision == "bf16" else None,
                                                 (st.stack32 if st.precision == "bf16" else st.stack).data_ptr(), n, M, self.frames,
                                                 st.head, self.obs.data_ptr(), done.data_ptr(), self.rows.data_ptr(), None,
                                                 _stream(self.device)), "ss_obs_stack_push_pool")
        self._blocks = blocks
        self._alloc_opp_stacks(self.pool_head)

    def rebalance_pool(self, weighting: str = "hard", p: float = 2.0, min_envs: int = 2, reset: bool = True) -> list:
        """Size each opponent's block by the learner's score against it: pool_progress(reset), pfsp_blocks of the scores
        (an opponent without finished games counts as 0.5), set_pool_blocks.  Returns the new blocks.  With per-env speeds
        each opponent was scored at the speeds of the envs its block covered; when the speeds are drawn independently per
        env (a random sweep), every block samples the same distribution and the scores stay comparable.  Sharded:
        collective; pool_progress sums the counters over the ranks and pfsp_blocks is deterministic, so every rank computes
        the same blocks."""
        prog = self.pool_progress(reset)
        blocks = pfsp_blocks([q["score"] if q["episodes"] else None for q in prog], self.pool_envs, weighting, p, min_envs)
        self.set_pool_blocks(blocks)
        return blocks

    def set_opponent(self, k: int, actor):
        """Replace opponent k of the pool with a copy of `actor` from the next tick on (the games in flight continue against
        it, with the slot's history), e.g. trainer.set_opponent(i % K, trainer.networks.actor) every few updates.  The actor
        must have the slot's frame count.  Sharded: collective; slot k then holds group rank 0's actor on every rank (one
        broadcast), and a refusal on any rank, or a different k, raises ValueError on every rank."""
        if self.opponents is None:
            raise ValueError("this trainer has no opponent pool")
        k, group = int(k), self.networks.group
        if group is None:
            v = self._opponent_vector(k, actor)
        else:
            refusal, v = None, None
            try:
                v = self._opponent_vector(k, actor)
            except (IndexError, ValueError) as e:
                refusal = str(e)
            ranks_agree(refusal, (("k", k),), group)
        self.opponents[k, :v.numel()].copy_(v)
        if group is not None:
            _broadcast_rank0(self.opponents[k], group)

    def _opponent_vector(self, k: int, actor) -> torch.Tensor:
        """`actor` as a flat vector for slot k (IndexError / ValueError when it does not fit the slot)."""
        if not 0 <= k < len(self.opponents):
            raise IndexError("opponent %d of %d" % (k, len(self.opponents)))
        f = self.opp_frames[k]
        n_params = int(lib.ss_actor_frames_params(f))
        if torch.is_tensor(actor) and actor.dim() == 1 and actor.numel() == n_params:
            return actor.detach()
        flat, frames = actor_vector(actor)
        if frames != f:
            raise ValueError("opponent %d has %d frames, the new actor %d" % (k, f, frames))
        return torch.from_numpy(flat)

    def pool_progress(self, reset: bool = False) -> list:
        """Per opponent, the training games against it finished so far (device counters): episodes, learner wins (the
        opponent was hit), learner losses, tick-limit endings (draws), mean episode ticks, and the learner's score with
        its standard error (win 1, draw 0.5, loss 0).  Sharded: collective; the figures are those of the counters summed
        over the ranks (one all-reduce), the same list on every rank, and `reset` zeroes each rank's own counters."""
        from .league import _score
        if self.opponents is None:
            raise ValueError("this trainer has no opponent pool")
        group = self.networks.group
        c = (self.pool_stats.cpu() if group is None else allreduce_counters(self.pool_stats, group)).numpy()
        if reset:
            self.pool_stats.zero_()
        out = []
        for k in range(c.shape[0]):
            games, wins, losses, draws, ticks = (int(v) for v in c[k, :5])
            score, se = _score(wins, draws, games)
            out.append(dict(episodes=games, wins=wins, losses=losses, draws=draws,
                            mean_ticks=ticks / games if games else float("nan"), score=score, stderr=se))
        return out

    def _rollout_pool(self, n_ticks: int, store: bool):
        """n_ticks ticks through ss_pool_rollout_frames (ss_pool_rollout_speeds when the envs have per-env speeds): the
        learner's forward, the opponents' forwards, the pool step and the history pushes."""
        envs, net, rp, st = self.envs, self.networks, self.replay, self.stack
        L, M, K = self.learner_rows, self.pool_envs, len(self.opponents)
        out = envs._buffers(1)
        a = _lib.PoolRolloutFramesArgs()
        a.state, a.n_envs, a.pool_envs, a.n_opponents = envs.state.data_ptr(), envs.n_envs, M, K
        a.params, a.opp_params, a.opp_param_stride = net.actor.data_ptr(), self.opponents.data_ptr(), self.opponents.shape[1]
        a.obs, a.act, a.reward = self.obs.data_ptr(), self.actions.data_ptr(), self._pool_reward.data_ptr()
        a.opp_obs, a.opp_act = self.obs[L:].data_ptr(), self.actions[L:].data_ptr()
        a.done, a.winner = out["done"].data_ptr(), out["winner"].data_ptr()
        if store:
            a.ring_obs, a.ring_act, a.ring_reward = rp.obs.data_ptr(), rp.act.data_ptr(), rp.reward.data_ptr()
            a.ring_next_obs, a.ring_done, a.capacity, a.write_pos = rp.next_obs.data_ptr(), rp.done.data_ptr(), rp.capacity, rp.pos
        a.n_ticks, a.param_noise_sd, a.noise_group, a.action_noise_sd = int(n_ticks), self.param_noise_sd, self.noise_group, 0.0
        a.tensor_cores, a.reward_mode, a.tick_limit = 1 if self.precision == "bf16" else 0, REWARD_MODES[envs.reward_mode], envs.tick_limit
        a.reset_mode = _lib.RESET_RANDOM if envs.random_positions else _lib.RESET_FIXED
        a.env_seed, a.env_counter, a.noise_seed, a.noise_counter = envs.seed, envs.counter, net.seed, net.counter
        a.status, a.step_flags = envs.status.data_ptr(), _lib.STEP_EPISODE_STATS if envs.collect_episode_stats else 0
        a.pool_stats = self.pool_stats.data_ptr()
        a.frames, a.head = self.frames, self.pool_head
        if st is not None:
            a.stack_tc = st.stack.data_ptr() if st.precision == "bf16" else None
            a.stack32 = (st.stack32 if st.precision == "bf16" else st.stack).data_ptr()
            a.rows = self.rows.data_ptr()
            a.noise_seed, a.noise_counter = st.seed, st.counter          # the stream FrameStackActor.forward draws from
        frames = (ctypes.c_int * K)(*self.opp_frames)
        stacks = (ctypes.c_void_p * K)(*[None if s is None else s.data_ptr() for s in self.opp_stacks])
        a.opp_frames, a.opp_stacks = frames, stacks
        table = None if self._blocks is None else (ctypes.c_int64 * K)(*self._blocks)
        a.opp_envs = table
        need = int(lib.ss_pool_rollout_frames_workspace_bytes(ctypes.byref(a)))
        if need > 0 and (self._pool_ws is None or self._pool_ws.numel() < need):
            self._pool_ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        if need > 0:
            a.workspace, a.workspace_bytes = self._pool_ws.data_ptr(), self._pool_ws.numel()
        with torch.cuda.device(self.device):
            if envs.speeds is not None:
                a.speeds = envs.speeds.data_ptr()
                check(lib.ss_pool_rollout_speeds(ctypes.byref(a), _stream(self.device)), "ss_pool_rollout_speeds")
            else:
                check(lib.ss_pool_rollout_frames(ctypes.byref(a), _stream(self.device)), "ss_pool_rollout_frames")
        envs.counter += n_ticks
        if st is None:
            net.counter += n_ticks
            self._pool_head += n_ticks
        else:
            st.head += n_ticks
            if self.param_noise_sd > 0:
                st.counter += n_ticks
        if store:
            rp.pos = (rp.pos + L * n_ticks) % rp.capacity
            rp.size = min(rp.capacity, rp.size + L * n_ticks)
        self.ticks += n_ticks
        return dict(obs=self.obs, reward=self._pool_reward, done=out["done"][0], winner=out["winner"][0])

    def rollout_tick(self, store: bool = True):
        """One tick of every env: actor forward on both players' observations (fresh parameter
        noise per noise group), env step, transition push."""
        self._ring_clean = False
        if self.opponents is not None:
            return self._rollout_pool(1, store)
        if self.frames > 1:
            return self._rollout_tick_frames(store)
        self.prev_obs, self.obs = self.obs, self.prev_obs
        self.networks.actor_forward(self.prev_obs, param_noise_sd=self.param_noise_sd, noise_group=self.noise_group,
                                    out=self.actions.view(-1, 2), precision=self.precision)
        out = self.envs.step(self.actions, obs_out=self.obs)
        if store:
            # the ring's flag masks the TD bootstrap: only a hit (winner != 0) is a termination, a tick-limit restart is not
            self.replay.push(self.prev_obs, self.actions, out["reward"], self.obs, out["winner"], done_div=2)
        self.ticks += 1
        return out

    def _rollout_tick_frames(self, store: bool = True):
        """The same tick for the frame-stacked networks: the actor reads each player's last `frames` observations; the stored
        transition is (stacked obs, action, reward, stacked obs after the tick, hit flag).  A restarted game's history is
        refilled with its first observation (FrameStackActor.push)."""
        st = self.stack
        st.forward(param_noise_sd=self.param_noise_sd, noise_group=self.noise_group if self.param_noise_sd > 0 else 0,
                   out=self.actions.view(-1, 2))
        out = self.envs.step(self.actions, obs_out=self.obs)
        st.push(self.obs.reshape(-1, 12), out["done"], done_div=2)
        self.prev_rows, self.rows = self.rows, self.prev_rows
        st.ordered_rows(out=self.rows)
        if store:
            self.replay.push(self.prev_rows, self.actions, out["reward"], self.rows, out["winner"], done_div=2)
        self.ticks += 1
        return out

    def rollout(self, n_ticks: int, store: bool = True):
        """n_ticks rollout ticks enqueued by ONE library call (ss_selfplay_rollout): same kernels and Philox
        counters as n_ticks calls of rollout_tick, without the per-tick host work."""
        self._ring_clean = False
        if self.opponents is not None:
            return self._rollout_pool(int(n_ticks), store)
        if self.frames > 1:
            for _ in range(int(n_ticks)):
                out = self._rollout_tick_frames(store)
            return dict(obs=self.obs, reward=out["reward"], done=out["done"], winner=out["winner"])
        envs, net, rp = self.envs, self.networks, self.replay
        if not envs.auto_reset:
            raise ValueError("the batched rollout needs auto_reset envs")
        if store and 2 * envs.n_envs > rp.capacity:
            raise ValueError("replay ring smaller than one tick of transitions")
        out = envs._buffers(1)
        # the current observation is in self.obs; it becomes buffer A of the call
        a, b = self.obs, self.prev_obs
        # SS_ROLLOUT_OVERLAP=1 (experiment, off by default): the env step runs beside the forward kernel on a second stream
        # (ss_selfplay_rollout2), consuming its actions tile by tile.  Bit-exact, and it works when both grids fit the GPU at
        # once; at 262,144 envs the forward kernel's CTAs fill their SMs (223 KB shared memory, 3/4 of the registers), the env
        # CTAs are not co-resident and their bounded waits expire (SS_STATUS_ROLLOUT_TIMEOUT) -- DESIGN.md section 6.5
        overlap = self.precision == "bf16" and os.environ.get("SS_ROLLOUT_OVERLAP", "0") == "1"
        if overlap and self._tile_ready is None:
            tiles = (2 * envs.n_envs + 127) // 128 + max(self.noise_group, 128) // 128 + 1
            self._tile_ready = torch.zeros(tiles, dtype=torch.int32, device=self.device)
            self._stream2 = torch.cuda.Stream(self.device, priority=-1)      # HIGHER priority than the current stream: the forward kernels
        with torch.cuda.device(self.device):
            check(lib.ss_selfplay_rollout2(
                envs.state.data_ptr(), envs.n_envs, net.actor.data_ptr(), a.data_ptr(), b.data_ptr(), self.actions.data_ptr(),
                out["reward"].data_ptr(), out["done"].data_ptr(), out["winner"].data_ptr(),
                rp.obs.data_ptr() if store else None, rp.act.data_ptr(), rp.reward.data_ptr(), rp.next_obs.data_ptr(),
                rp.done.data_ptr(), rp.capacity, rp.pos, int(n_ticks), self.param_noise_sd, self.noise_group, 0.0,
                1 if self.precision == "bf16" else 0, REWARD_MODES[envs.reward_mode], envs.tick_limit,
                _lib.RESET_RANDOM if envs.random_positions else _lib.RESET_FIXED, envs.seed, envs.counter, net.seed,
                net.counter, _ptr(envs.speeds), envs.status.data_ptr(), _lib.STEP_EPISODE_STATS if envs.collect_episode_stats else 0,
                self._tile_ready.data_ptr() if overlap else None, self._stream2.cuda_stream if overlap else None,
                _stream(self.device)), "ss_selfplay_rollout")
        envs.counter += n_ticks
        net.counter += n_ticks
        if store:
            rp.pos = (rp.pos + 2 * envs.n_envs * n_ticks) % rp.capacity
            rp.size = min(rp.capacity, rp.size + 2 * envs.n_envs * n_ticks)
        rows = 2 * envs.n_envs
        in_place = (store and rp.capacity % rows == 0 and (rp.pos - rows * n_ticks) % rows == 0
                    and (rp.capacity // rows >= 2 or n_ticks == 1))       # the library's own condition (ss_selfplay_rollout)
        if (n_ticks & 1) and not in_place:        # (in place, the library leaves the current observation in buffer A)
            self.obs, self.prev_obs = b, a
        self.ticks += n_ticks
        return dict(obs=self.obs, reward=out["reward"][0], done=out["done"][0], winner=out["winner"][0])

    # -- checkpoint / resume (SkillshotLearner.py:123-162 keeps the two Keras models; a batched run also needs the
    #    optimiser moments, the targets, the games in flight, the replay ring and every Philox counter) ---------------
    def state_dict(self):
        sd = dict(envs=self.envs.state_dict(), networks=self.networks.state_dict(), replay=self.replay.state_dict(),
                  obs=self.obs.cpu(), actions=self.actions.cpu(), ticks=self.ticks, batch_size=self.batch_size,
                  param_noise_sd=self.param_noise_sd, noise_group=self.noise_group, precision=self.precision, frames=self.frames,
                  update_precision=self.update_precision)
        if self.stack is not None:      # the players' observation histories and the noise stream of the stacked actor
            st = self.stack
            sd["stack"] = dict(stack=st.stack.cpu(), stack32=None if st.stack32 is None else st.stack32.cpu(), head=st.head,
                               counter=st.counter, seed=st.seed, rows=self.rows.cpu())
        if self.opponents is not None:
            sd["pool"] = dict(opponents=self.opponents.cpu(), pool_envs=self.pool_envs, stats=self.pool_stats.cpu(),
                              frames=list(self.opp_frames), stacks=[None if s is None else s.cpu() for s in self.opp_stacks],
                              head=self.pool_head, blocks=None if self._blocks is None else list(self._blocks))
        return sd

    def load_state_dict(self, sd):
        pool = sd.get("pool")            # absent: a trainer without a pool
        have = (0, 0) if self.opponents is None else (self.pool_envs, len(self.opponents), self.frames, tuple(self.opp_frames))
        want = (0, 0)
        if pool is not None:             # (a checkpoint of a pool of 1-frame actors may lack the frame counts)
            K = int(pool["opponents"].shape[0])
            want = (int(pool["pool_envs"]), K, int(sd.get("frames", 1)), tuple(int(f) for f in pool.get("frames", [1] * K)))
        if have != want:
            raise ValueError("checkpoint pool layout (pool_envs, opponents, frames, opponent frames) = %s, this trainer's %s"
                             % (want, have))
        self.networks.check_state_dict(sd["networks"])
        self.envs.load_state_dict(sd["envs"])
        self.networks.load_state_dict(sd["networks"])
        self.replay.load_state_dict(sd["replay"])
        self.obs.copy_(sd["obs"].to(self.device))
        self.actions.copy_(sd["actions"].to(self.device))
        self.ticks, self.batch_size = int(sd["ticks"]), int(sd["batch_size"])
        self.param_noise_sd, self.noise_group = float(sd["param_noise_sd"]), int(sd["noise_group"])
        self.update_precision = sd.get("update_precision")      # absent from older checkpoints: None
        if self.stack is not None:
            st, ss = self.stack, sd["stack"]
            st.stack.copy_(ss["stack"].to(self.device))
            if st.stack32 is not None:
                st.stack32.copy_(ss["stack32"].to(self.device))
            st.head, st.counter = int(ss["head"]), int(ss["counter"])
            st.seed = int(ss.get("seed", st.seed))       # (absent from older checkpoints: this trainer's seed)
            self.rows.copy_(ss["rows"].to(self.device))
        if pool is not None:
            # the blocks are run state: adopt the checkpoint's (absent: M / K each), with histories of its sizes
            blocks = pool.get("blocks")
            self._blocks = None if blocks is None else check_pool_blocks(blocks, self.pool_envs, len(self.opponents))
            self._alloc_opp_stacks(0, fill=False)
            self.opponents.copy_(pool["opponents"].to(self.device))
            self.pool_stats.copy_(pool["stats"].to(self.device))
            for s, saved in zip(self.opp_stacks, pool.get("stacks", [None] * len(self.opp_stacks))):
                if s is not None:
                    s.copy_(saved.to(self.device))
            if self.stack is None:      # (a frame-stacked learner's counter came back with its history)
                self._pool_head = int(pool.get("head", 0))
        self._batch = None
        self._batches = [None, None]
        self._ring_clean = False

    def record_boards(self, env: int, n_ticks: int, path: Optional[str] = None, store: bool = True):
        """Play n_ticks rollout ticks and return the 250 x 250 rasters of game `env` after each of them
        (SkillshotGame.get_board, SkillshotGame.py:36-56, rebuilt on the host from the exported state row): the frames
        SkillshotGameDisplay.display_sequence shows.  With `path`, also written as training_boards.npy in the shape
        save_training_boards uses (one object-array entry = one sequence, SkillshotLearner.py:182-204)."""
        from .game import render_board
        boards = []
        for _ in range(int(n_ticks)):
            self.rollout_tick(store=store)
            boards.append(render_board(self.envs.export_state(int(env), 1), 0))
        boards = np.asarray(boards)
        if path is not None:
            os.makedirs(path, exist_ok=True)
            arr = np.empty(1, dtype=object)
            arr[0] = boards
            np.save(os.path.join(path, "training_boards"), arr, allow_pickle=True)
        return boards

    def progress(self, reset: bool = False) -> dict:
        """The training-progress log of the reference (per-episode ticks and winner, SkillshotLearner.py:164-180,
        365-366) for the games finished so far, reduced on the device by the step kernel (SkillshotEnvs.episode_summary)."""
        return self.envs.episode_summary(reset=reset)

    def evaluate(self, opponent, n_games: int = 65536, seed: int = 0, tick_limit: Optional[int] = None) -> dict:
        """Play the current actor (with this trainer's frames and `precision`) against `opponent` -- a flat actor vector or
        the six get_weights() arrays, see Match -- over n_games seat-balanced games and return Match.play's result
        (score is the current actor's).  The tick limit (default: the trainer's), start mode and per-env speeds (env j
        takes those of the trainer's env j mod n_envs) are the trainer's.  The match has its own envs, buffers and Philox
        stream and copies the actor: the trainer's envs, ring, networks and counters are not touched, so a run that
        evaluates in the middle continues bit-identically."""
        envs = self.envs
        limit = envs.tick_limit if tick_limit is None else int(tick_limit)
        if limit <= 0:
            raise ValueError("a match needs a positive tick_limit (the trainer has none)")
        speeds = None
        if envs.speeds is not None:
            n, buf = envs.n_envs, envs.speeds
            idx = torch.arange(int(n_games), device=self.device) % n
            f = buf[:16 * n].view(torch.float64).view(n, 2)
            g = buf[16 * n:]
            speeds = (f[idx, 0], f[idx, 1], g.view(torch.float64).view(n, 2)[idx, 0], g.view(torch.int64).view(n, 2)[idx, 1])
        return Match(self.networks.actor, opponent, n_games, device=self.device, precision=self.precision, tick_limit=limit,
                     random_positions=envs.random_positions, seed=seed, speeds=speeds).play()

    def evaluate_league(self, opponents, games_per_pair: int = 8192, seed: int = 0, tick_limit: Optional[int] = None) -> dict:
        """Play the current actor (policy 0, with this trainer's frames and `precision`) against each of `opponents` (flat
        actor vectors or six get_weights() arrays, see League) in a gauntlet of games_per_pair seat-balanced games per
        opponent and return League.play's result (ratings: the current actor's is ratings[0]).  The tick limit (default:
        the trainer's), start mode and per-env speeds (league env j takes those of the trainer's env j mod n_envs) are the
        trainer's, as in evaluate().  The league has its own envs, buffers and Philox stream and copies every actor: the
        trainer's envs, ring, networks and counters are not touched."""
        from .league import League, gauntlet
        envs = self.envs
        limit = envs.tick_limit if tick_limit is None else int(tick_limit)
        if limit <= 0:
            raise ValueError("a league needs a positive tick_limit (the trainer has none)")
        actors = [self.networks.actor] + list(opponents)
        n_games = (len(actors) - 1) * int(games_per_pair)
        speeds = None
        if envs.speeds is not None:
            n, buf = envs.n_envs, envs.speeds
            idx = torch.arange(n_games, device=self.device) % n
            f = buf[:16 * n].view(torch.float64).view(n, 2)
            g = buf[16 * n:]
            speeds = (f[idx, 0], f[idx, 1], g.view(torch.float64).view(n, 2)[idx, 0], g.view(torch.int64).view(n, 2)[idx, 1])
        return League(actors, games_per_pair, pairs=gauntlet(len(actors)), device=self.device, precision=self.precision,
                      tick_limit=limit, random_positions=envs.random_positions, seed=seed, speeds=speeds).play()

    def check_exchange(self):
        """Raises if a rank's gradient failed to arrive in the fused peer exchange (the Adam kernels skip their writes from
        that point on, so the ranks still hold identical weights: reload or stop)."""
        if self.networks.peer is not None:
            self.networks.peer.check_status()

    def save(self, path: str):
        """Write a checkpoint the run can be resumed from bit-identically (one file per rank when sharded)."""
        self.check_exchange()
        torch.cuda.synchronize(self.device)
        os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
        torch.save(self.state_dict(), path)

    def load(self, path: str):
        self.load_state_dict(torch.load(path, map_location="cpu", weights_only=False))

    def update(self):
        """One critic step and one actor step on a sampled minibatch: a single library call on one GPU or
        with the fused peer exchange, the separate steps (update_stepwise) around an NCCL all-reduce, for frames > 1 and
        for the TD3 update (any of the four TD3 options not at its default)."""
        net = self.networks
        if (net.group is not None and net.peer is None) or self.frames > 1 or net.td3:
            return self.update_stepwise()
        # two sets of minibatch buffers in turn: when no rollout has touched the ring since the previous update, this
        # update's rows are drawn while that update's last kernels still run (ss_ddpg_update_args.sample_early)
        k = self.updates & 1
        # (measured, profiles/r2_update_sample_early_ab.txt: 158.1 -> 152.1 us at 65,536 rows; at 524,288 rows the gather
        #  competes with what it runs beside, 759 -> 764 us: small minibatches only)
        early = self._ring_clean and self._batches[k] is not None and self.batch_size <= 131072
        self._batch = self._batches[k] = net.update_from_ring(self.replay, self.batch_size, out=self._batches[k], sample_early=early)
        self._ring_clean = True
        self.updates += 1
        if net.peer is not None and self.updates % self.exchange_check_every == 0:
            net.peer.check_status()         # one device-to-host read every few hundred updates
        return net.stats[0], net.stats[1]

    def update_stepwise(self):
        """The same update as one library call per step (sample, target, critic step, actor step); with the TD3 options,
        ActorCritic.td3_step on the minibatch."""
        self._ring_clean = False
        self._batch = b = self.replay.sample(self.batch_size, out=self._batch)
        net = self.networks
        if net.td3:
            return net.td3_step(b["obs"], b["act"], b["reward"], b["next_obs"], b["done"])
        y = net.td_targets(b["reward"], b["next_obs"], b["done"])
        sse = net.critic_step(b["obs"], b["act"], y)
        q = net.actor_step(b["obs"])
        return sse, q
