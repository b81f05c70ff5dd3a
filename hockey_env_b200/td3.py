"""Device-side TD3 update and prioritized replay fed straight from the batched env -- SURVEY.md section 8f rank 3.

What the reference does one transition and one host round trip at a time (rl/td3/learner.py:55-219,
rl/replay/prioritized_buffer.py:6-69, rl/td3/networks.py:36-70, rl/td3/config.py) is done here on whole device batches:
the replay buffer lives in HBM, sampling / importance weights / priority updates never leave the device, and the
learner consumes the sampled tensors in place.  Same algorithm, same hyper-parameter names and defaults.  The networks
are plain torch modules (library GEMMs + autograd): they are the dense ops next to the env path, not the path.
"""
import copy
import math
from dataclasses import dataclass

import torch
from torch import nn

from .actor import ActorNetwork
from .training import DeviceReplayBuffer


@dataclass
class TD3Config:
    """The reference's TD3Config fields that the update uses (rl/td3/config.py), same defaults."""
    gamma: float = 0.99
    tau_actor: float = 0.005
    tau_critic: float = 0.005
    policy_update_freq: int = 2
    lr_q: float = 4e-4
    lr_pol: float = 4e-4
    wd_q: float = 0.0
    wd_pol: float = 0.0
    prioritized_replay: bool = False
    beta: float = 0.15
    buffer_size: int = 300_000
    batch_size: int = 256
    action_noise_scale: float = 0.2
    target_action_noise_scale: float = 0.2
    target_action_noise_clip: float = 0.3


class QNetwork(nn.Module):
    def __init__(self, in_dim, hidden):
        super().__init__()
        self.fc1 = nn.Linear(in_dim, hidden)
        self.fc2 = nn.Linear(hidden, hidden)
        self.fc3 = nn.Linear(hidden, 1)

    def forward(self, x):
        return self.fc3(torch.tanh(self.fc2(torch.tanh(self.fc1(x)))))


class TwinQNetwork(nn.Module):
    """Two independent Q heads on [obs, action] (rl/td3/networks.py:36-70: each head is the reference's 3-layer tanh MLP
    with a linear output; state_dict keys q1.fc*/q2.fc* and the action_low/high/range buffers match its checkpoints)."""

    def __init__(self, obs_dim=18, action_dim=4, hidden=256):
        super().__init__()
        self.register_buffer("action_low", -torch.ones(action_dim))
        self.register_buffer("action_high", torch.ones(action_dim))
        self.register_buffer("action_range", 2 * torch.ones(action_dim))
        self.q1 = QNetwork(obs_dim + action_dim, hidden)
        self.q2 = QNetwork(obs_dim + action_dim, hidden)

    def forward(self, obs, action):
        if not torch.isinf(self.action_range).any():  # actions normalised to [-1, 1] (identity for this env's bounds)
            action = (action - self.action_low) / self.action_range * 2 - 1.0
        x = torch.cat([obs, action], dim=-1)
        return self.q1(x).squeeze(-1), self.q2(x).squeeze(-1)


def huber_weighted(x, y, weights=None):
    """rl/utils/torch_utils.py:12-24: smooth-L1 with per-sample weights, mean over the batch."""
    d = x - y
    w = torch.ones_like(d) if weights is None else weights
    return torch.where(d.abs() < 1, 0.5 * w * d * d, (d.abs() - 0.5) * w).mean()


class DevicePrioritizedReplayBuffer(DeviceReplayBuffer):
    """Proportional prioritized replay on the device (rl/replay/prioritized_buffer.py:6-69): a new transition gets the
    current maximum weight (1e8 while the buffer is empty), sampling is proportional to the weights, the learner writes
    the clamped TD errors back as the new weights of the batch it just used."""

    def __init__(self, capacity, obs_dim=18, action_dim=4, device="cuda:0", seed=0, init_weight=1e8):
        super().__init__(capacity, obs_dim, action_dim, device, seed)
        self.init_weight = float(init_weight)
        self.weights = torch.full((self.capacity,), self.init_weight, dtype=torch.float32, device=self.device)
        self.last_batch_inds = None

    def push(self, obs, action, reward, next_obs, done):
        n = obs.shape[0]
        top = self.weights[:self.size].max() if self.size > 0 else torch.tensor(self.init_weight, device=self.device)
        start = self.pos
        super().push(obs, action, reward, next_obs, done)
        idx = (start + torch.arange(n, device=self.device)) % self.capacity
        self.weights[idx] = top

    def sample_indices(self, batch_size):
        """Draw min(batch_size, len) indices proportionally to the weights; they become `last_batch_inds`."""
        batch_size = min(int(batch_size), self.size)
        w = torch.nan_to_num(self.weights[:self.size], nan=0.0, posinf=0.0, neginf=0.0).clamp_min(1e-6)
        idx = torch.multinomial(w / w.sum(), batch_size, replacement=True, generator=self.gen)
        self.last_batch_inds = idx
        return idx

    def sample(self, batch_size):
        idx = self.sample_indices(batch_size)
        return self.obs[idx], self.action[idx], self.reward[idx], self.next_obs[idx], self.done[idx]

    def get_last_probs(self):
        p = self.weights[self.last_batch_inds]
        tot = p.sum()
        return p / tot if float(tot) > 0 else torch.full_like(p, 1.0 / p.numel())

    def update_priorities(self, priorities):
        self.weights[self.last_batch_inds] = priorities.to(self.weights.dtype)
        self.last_batch_inds = None


class PopulationReplayBuffer:
    """One device replay buffer for a population of K learners (`FusedTD3Population`): arrays of K * capacity rows, of
    which member m owns rows [m * capacity, (m + 1) * capacity), each a ring buffer like `DeviceReplayBuffer` (or, with
    prioritized=True, like `DevicePrioritizedReplayBuffer`).  All members share the ring position and the size.

    `push` takes the transitions of N = K * n envs: env block m (rows [m * n, (m + 1) * n)) goes to member m, one strided
    copy per array.  `sample_indices(b)` returns [K, b] int64 GLOBAL rows, member m's inside its own rows, so that one
    population update reads all members' batches from the shared arrays (and, prioritized, writes each member's
    priorities into its own rows only)."""

    def __init__(self, k, capacity, obs_dim=18, action_dim=4, device="cuda:0", seed=0, prioritized=False, init_weight=1e8):
        self.k, self.capacity, self.device = int(k), int(capacity), torch.device(device)
        if self.k < 1 or self.capacity < 1:
            raise ValueError("PopulationReplayBuffer needs k >= 1 and capacity >= 1")
        rows = self.k * self.capacity
        self.obs = torch.empty((rows, obs_dim), dtype=torch.float32, device=self.device)
        self.action = torch.empty((rows, action_dim), dtype=torch.float32, device=self.device)
        self.reward = torch.empty(rows, dtype=torch.float32, device=self.device)
        self.next_obs = torch.empty((rows, obs_dim), dtype=torch.float32, device=self.device)
        self.done = torch.empty(rows, dtype=torch.float32, device=self.device)
        self.prioritized = bool(prioritized)
        self.init_weight = float(init_weight)
        self.weights = torch.full((rows,), self.init_weight, dtype=torch.float32, device=self.device) if self.prioritized else None
        self.pos, self.size = 0, 0
        self.seed = seed
        self.gen = torch.Generator(device=self.device)
        self.gen.manual_seed(seed)
        self.offsets = torch.arange(self.k, dtype=torch.int64, device=self.device).unsqueeze(1) * self.capacity  # [K, 1]

    def __len__(self):
        return self.size

    def _rows(self, t):
        """[K, capacity, ...] view of a [K * capacity, ...] array."""
        return t.view(self.k, self.capacity, *t.shape[1:])

    def push(self, obs, action, reward, next_obs, done):
        """N = K * n transitions (n <= capacity); block m of the batch goes to member m's ring."""
        n_all = obs.shape[0]
        if n_all % self.k:
            raise ValueError(f"PopulationReplayBuffer.push: {n_all} rows do not split into {self.k} equal blocks")
        n = n_all // self.k
        if n > self.capacity:
            raise ValueError("batch larger than the buffer")
        top = None
        if self.prioritized:
            w = self._rows(self.weights)
            top = w[:, :self.size].amax(1) if self.size > 0 else torch.full((self.k,), self.init_weight, device=self.device)
        first = min(n, self.capacity - self.pos)
        for dst, src in ((self.obs, obs), (self.action, action), (self.reward, reward), (self.next_obs, next_obs),
                         (self.done, done.to(torch.float32))):
            d, sv = self._rows(dst), src.reshape(self.k, n, *src.shape[1:])
            d[:, self.pos:self.pos + first].copy_(sv[:, :first])
            if first < n:
                d[:, :n - first].copy_(sv[:, first:])
        if top is not None:
            w = self._rows(self.weights)
            w[:, self.pos:self.pos + first] = top.unsqueeze(1)
            if first < n:
                w[:, :n - first] = top.unsqueeze(1)
        self.pos = (self.pos + n) % self.capacity
        self.size = min(self.capacity, self.size + n)

    def sample_indices(self, batch_size):
        """[K, b] int64 global rows, b = min(batch_size, len): uniform over each member's stored rows (one randint), or
        proportional to each member's weights (one row-wise multinomial)."""
        b = min(int(batch_size), self.size)
        if not self.prioritized:
            local = torch.randint(0, self.size, (self.k, b), device=self.device, generator=self.gen)
        else:
            w = torch.nan_to_num(self._rows(self.weights)[:, :self.size], nan=0.0, posinf=0.0, neginf=0.0).clamp_min(1e-6)
            local = torch.multinomial(w / w.sum(1, keepdim=True), b, replacement=True, generator=self.gen)
        return local + self.offsets

    def member(self, m):
        """Member m's rows as a `DeviceReplayBuffer` (prioritized: `DevicePrioritizedReplayBuffer`) over VIEWS of this
        buffer's arrays, with this buffer's current size and position and a generator of its own (seeded seed + 1 + m).
        Writes through either alias the same memory; size and position are copied, not shared."""
        m = int(m)
        if not 0 <= m < self.k:
            raise IndexError(f"member {m} out of range [0, {self.k})")
        cls = DevicePrioritizedReplayBuffer if self.prioritized else DeviceReplayBuffer
        out = cls.__new__(cls)
        out.capacity, out.device = self.capacity, self.device
        lo, hi = m * self.capacity, (m + 1) * self.capacity
        out.obs, out.action, out.reward = self.obs[lo:hi], self.action[lo:hi], self.reward[lo:hi]
        out.next_obs, out.done = self.next_obs[lo:hi], self.done[lo:hi]
        out.pos, out.size = self.pos, self.size
        out.gen = torch.Generator(device=self.device)
        out.gen.manual_seed(self.seed + 1 + m)
        if self.prioritized:
            out.init_weight, out.weights, out.last_batch_inds = self.init_weight, self.weights[lo:hi], None
        return out


class DeviceTD3Learner:
    """TD3Learner.update (rl/td3/learner.py:55-219) on device batches: clipped-noise target actions, min of the twin target
    critics, weighted smooth-L1 critic loss (mean of both heads), actor and Polyak target updates every
    `policy_update_freq` critic steps, and -- with a prioritized buffer -- importance weights (1 / (N p))^beta
    normalised by their maximum and |TD| priorities clamped to [1e-6, 1e6]."""

    def __init__(self, actor=None, critic=None, config=None, replay_buffer=None, device="cuda:0", seed=0):
        self.cfg = config or TD3Config()
        self.device = torch.device(device)
        self.actor = (actor or ActorNetwork()).to(self.device)
        self.critic = (critic or TwinQNetwork()).to(self.device)
        self.target_actor = copy.deepcopy(self.actor).requires_grad_(False)
        self.target_critic = copy.deepcopy(self.critic).requires_grad_(False)
        self.actor_optimizer = torch.optim.Adam(self.actor.parameters(), lr=self.cfg.lr_pol, weight_decay=self.cfg.wd_pol)
        self.critic_optimizer = torch.optim.Adam(self.critic.parameters(), lr=self.cfg.lr_q, weight_decay=self.cfg.wd_q)
        self.replay_buffer = replay_buffer
        self.prioritized = isinstance(replay_buffer, DevicePrioritizedReplayBuffer)
        self.train_step = 0
        self.gen = torch.Generator(device=self.device)
        self.gen.manual_seed(seed)
        self.seed = seed
        self.fused_actor = None  # train(..., fused=True): the FusedActor mirror of `actor` that acts in the env

    @torch.no_grad()
    def compute_target(self, next_state, reward, done):
        a = self.target_actor(next_state)
        noise = torch.randn(a.shape, device=a.device, generator=self.gen) * self.cfg.target_action_noise_scale
        noise = noise.clamp(-self.cfg.target_action_noise_clip, self.cfg.target_action_noise_clip)
        a = (a + noise).clamp(-1.0, 1.0)
        q1, q2 = self.target_critic(next_state, a)
        return reward + self.cfg.gamma * (1 - done.float()) * torch.minimum(q1, q2)

    def importance_weights(self):
        if not self.prioritized or self.replay_buffer.last_batch_inds is None:
            return None
        probs = self.replay_buffer.get_last_probs()
        w = (1.0 / (probs * self.replay_buffer.size)) ** self.cfg.beta
        top = w.max()
        return w / top if float(top) > 0 else w

    def update(self, state, action, reward, next_state, done):
        """One learner step on a batch; returns (actor_loss or None, critic_loss) as device scalars (no host sync)."""
        self.train_step += 1
        target = self.compute_target(next_state, reward, done)
        self.critic_optimizer.zero_grad(set_to_none=True)
        q1, q2 = self.critic(state, action)
        weights = self.importance_weights()
        critic_loss = 0.5 * (huber_weighted(q1, target, weights) + huber_weighted(q2, target, weights))
        critic_loss.backward()
        self.critic_optimizer.step()
        if self.prioritized and self.replay_buffer.last_batch_inds is not None:
            td = 0.5 * ((q1 - target).abs() + (q2 - target).abs())
            self.replay_buffer.update_priorities(td.detach().clamp(1e-6, 1e6))
        actor_loss = None
        if self.train_step % self.cfg.policy_update_freq == 0:
            self.actor_optimizer.zero_grad(set_to_none=True)
            q, _ = self.critic(state, self.actor(state))
            actor_loss = -q.mean()
            actor_loss.backward()
            self.actor_optimizer.step()
            self._polyak(self.actor, self.target_actor, self.cfg.tau_actor)
            self._polyak(self.critic, self.target_critic, self.cfg.tau_critic)
            actor_loss = actor_loss.detach()
        return actor_loss, critic_loss.detach()

    def update_from_buffer(self, batch_size=None):
        return self.update(*self.replay_buffer.sample(batch_size or self.cfg.batch_size))

    @staticmethod
    @torch.no_grad()
    def _polyak(net, target, tau):
        for tp, p in zip(target.parameters(), net.parameters()):
            tp.mul_(1 - tau).add_(p, alpha=tau)

    # checkpoints in the reference's format (TD3Agent.save / load, rl/td3/agent.py:269-284)
    def state_dict(self):
        return {"policy": self.actor.state_dict(), "critic": self.critic.state_dict(),
                "target_policy": self.target_actor.state_dict(), "target_critic": self.target_critic.state_dict()}

    def load_state_dict(self, ckpt):
        self.actor.load_state_dict(ckpt["policy"])
        self.critic.load_state_dict(ckpt["critic"])
        self.target_actor.load_state_dict(ckpt["target_policy"])
        self.target_critic.load_state_dict(ckpt["target_critic"])


_ACTOR_SHAPES = {"fc1.weight": (256, 18), "fc1.bias": (256,), "fc2.weight": (256, 256), "fc2.bias": (256,),
                 "fc3.weight": (4, 256), "fc3.bias": (4,)}
_HEAD_SHAPES = {"fc1.weight": (256, 22), "fc1.bias": (256,), "fc2.weight": (256, 256), "fc2.bias": (256,),
                "fc3.weight": (1, 256), "fc3.bias": (1,)}
_CRITIC_SHAPES = {f"{h}.{k}": v for h in ("q1", "q2") for k, v in _HEAD_SHAPES.items()}


def _pad64(n):
    return (n + 63) // 64 * 64


class FusedTD3Learner(DeviceTD3Learner):
    """`DeviceTD3Learner.update` as ONE sm_100a kernel launch per update (csrc/hk_td3.cuh, hk_td3_update): the batch
    gather, the target policy with clipped smoothing noise, the twin-critic step with Adam, prioritized importance
    weights and priority write-back, and on actor steps the actor step and the Polyak updates.  No host sync, no
    allocation in the kernel call; graph-capturable.  fp32 throughout with fixed summation orders: bit-reproducible run
    to run, and equal to the torch learner up to fp32 rounding (not bit for bit).

    Every parameter of actor, critic, target_actor and target_critic is re-homed into a view of one device arena, so the
    modules, `state_dict()` / `load_state_dict()` (the reference's checkpoint format, interchangeable with
    `DeviceTD3Learner`) and `FusedActor.refresh(learner.actor)` work on the live weights.  The Adam state lives in the
    arena as well, with its step counts as device int64: `actor_optimizer` / `critic_optimizer` exist but are never
    stepped, and checkpoints carry no optimizer state, as in the reference.  The target-policy noise is Philox keyed on
    (seed, batch row, a device counter that every update advances), not torch's generator; the replay indices still come
    from the buffer's generator (`sample_indices`), so a fused and a torch learner on equal buffers train on the same
    batches.  Only the reference architecture is supported (actor 18-256-256-4, critic 22-256-256-1), on CUDA.  The
    kernel normalises both critics' actions with the critic's action bounds, so a checkpoint whose target critic carries
    other action_low / action_range buffers is rejected with ValueError."""

    MAX_BATCH = 1024

    def __init__(self, actor=None, critic=None, config=None, replay_buffer=None, device="cuda:0", seed=0, arena=None):
        """arena: None (allocate one), or a zeroed contiguous uint8 CUDA tensor of hk_td3_arena_bytes() bytes on `device`
        to home the parameters in (FusedTD3Population passes rows of its [K, bytes] arena table)."""
        import ctypes as C
        from . import _lib
        from .actor import _cuda_device
        super().__init__(actor, critic, config, replay_buffer, device, seed)
        self.device = _cuda_device(self.device, "FusedTD3Learner")
        self._C, self._lib = C, _lib
        self.L = _lib.load()
        for net, shapes, who in ((self.actor, _ACTOR_SHAPES, "actor"), (self.critic, _CRITIC_SHAPES, "critic")):
            got = {k: tuple(v.shape) for k, v in net.named_parameters()}
            if got != shapes:
                raise ValueError(f"FusedTD3Learner implements the reference architecture only (actor 18-256-256-4, twin "
                                 f"critic 22-256-256-1); the {who} has parameters {got}")
        self._check_action_bounds(self.critic.state_dict(), self.target_critic.state_dict())
        blocks, ctr_off, nbytes = self.arena_layout()
        if nbytes != int(self.L.hk_td3_arena_bytes()):
            raise _lib.HockeyLibraryError("FusedTD3Learner: the library's arena size does not match this package")
        if arena is None:
            arena = torch.zeros(nbytes, dtype=torch.uint8, device=self.device)
        elif not (arena.dtype == torch.uint8 and arena.is_contiguous() and tuple(arena.shape) == (nbytes,)
                  and arena.device == self.device and arena.data_ptr() % 16 == 0):
            raise ValueError(f"FusedTD3Learner: arena must be a contiguous 16-byte aligned uint8 tensor [{nbytes}] on {self.device}")
        self.arena = arena
        f = self.arena.view(torch.float32)
        self.blocks = {name: f[o:o + n] for name, (o, n) in blocks.items()}  # flat fp32 views, parameters in state_dict order
        self.counters = self.arena[4 * ctr_off:4 * ctr_off + 24].view(torch.int64)  # critic step, actor step, noise counter
        for name, net in (("actor", self.actor), ("critic", self.critic), ("target_actor", self.target_actor),
                          ("target_critic", self.target_critic)):
            blk, o = self.blocks[name], 0
            with torch.no_grad():
                for p in net.parameters():  # state_dict order without the critic's buffers
                    view = blk[o:o + p.numel()].view(p.shape)
                    view.copy_(p.detach().to(torch.float32))
                    p.data = view
                    o += p.numel()
        self._losses = None
        self._scratch, self._scratch_b = None, 0
        self._arange = None
        self._hp = _lib.TD3HParams()

    @staticmethod
    def arena_layout():
        """The arena of include/hockey_b200.h (hk_td3_update): ({block: (float offset, floats)}, float offset of the three
        int64 counters, bytes).  Blocks start at multiples of 64 floats."""
        pa = sum(math.prod(s) for s in _ACTOR_SHAPES.values())
        pc = sum(math.prod(s) for s in _CRITIC_SHAPES.values())
        blocks, off = {}, 0
        for name, n in (("actor", pa), ("critic", pc), ("target_actor", pa), ("target_critic", pc), ("m_actor", pa),
                        ("v_actor", pa), ("m_critic", pc), ("v_critic", pc)):
            blocks[name] = (off, n)
            off += _pad64(n)
        return blocks, off, 4 * (off + 64)

    @staticmethod
    def _check_action_bounds(critic_sd, target_sd):
        """The kernel normalises the target critic's actions with the critic's action_low / action_range buffers, so the
        two critics must carry equal ones (DeviceTD3Learner would use the target critic's own)."""
        for k in ("action_low", "action_range"):
            if not torch.equal(critic_sd[k].detach().cpu(), target_sd[k].detach().cpu()):
                raise ValueError(f"FusedTD3Learner: the critic's and the target critic's {k} differ "
                                 f"({critic_sd[k].tolist()} vs {target_sd[k].tolist()}); the fused update uses the critic's")

    def load_state_dict(self, ckpt):
        self._check_action_bounds(ckpt["critic"], ckpt["target_critic"])
        super().load_state_dict(ckpt)

    def _hparams(self):
        c, hp = self.cfg, self._hp
        for k, v in (("gamma", c.gamma), ("tau_actor", c.tau_actor), ("tau_critic", c.tau_critic), ("lr_actor", c.lr_pol),
                     ("lr_critic", c.lr_q), ("wd_actor", c.wd_pol), ("wd_critic", c.wd_q), ("beta", c.beta),
                     ("target_noise", c.target_action_noise_scale), ("target_noise_clip", c.target_action_noise_clip)):
            setattr(hp, k, float(v))
        return hp

    def _launch(self, arrays, idx, prio):
        """One hk_td3_update on the current stream; arrays = (obs, action, reward, next_obs, done) base tensors, idx their
        int64 rows, prio = (weights, weight indices, N) or None."""
        C = self._C
        b = idx.shape[0]
        if not 1 <= b <= self.MAX_BATCH:
            raise ValueError(f"FusedTD3Learner: batch size must be in [1, {self.MAX_BATCH}], got {b}")
        if self._scratch is None or self._scratch_b < b:
            self._scratch = torch.empty(int(self.L.hk_td3_scratch_bytes(b)), dtype=torch.uint8, device=self.device)
            self._scratch_b = b
        self.train_step += 1
        do_actor = self.train_step % self.cfg.policy_update_freq == 0
        losses = torch.empty(2, dtype=torch.float32, device=self.device)
        batch = self._lib.TD3Batch(*[t.data_ptr() for t in arrays], idx.data_ptr())
        if prio is not None:
            batch.prio_weights, batch.prio_idx, batch.prio_n = prio[0].data_ptr(), prio[1].data_ptr(), int(prio[2])
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            self._lib.check(self.L.hk_td3_update(
                C.c_void_p(self.arena.data_ptr()), C.c_void_p(self._scratch.data_ptr()), C.byref(batch), b, C.byref(self._hparams()),
                C.c_void_p(self.critic.action_low.data_ptr()), C.c_void_p(self.critic.action_range.data_ptr()),
                self.seed & (2**64 - 1), int(do_actor), C.c_void_p(losses.data_ptr()), self.device.index or 0, C.c_void_p(stream)))
        self._last_batch = b
        return (losses[0] if do_actor else None), losses[1]

    def last_importance_weights(self):
        """[B] importance weights the last update used (ones for a uniform batch), computed in the kernel."""
        return self._scratch.view(torch.float32)[:self._last_batch]

    @staticmethod
    def _f32(t):
        return t.detach().to(torch.float32).contiguous()

    def update(self, state, action, reward, next_state, done):
        """One learner step on a given batch, in one launch; returns (actor_loss or None, critic_loss) as device scalars.
        With a prioritized buffer whose `last_batch_inds` are set (the batch came from its `sample`), the importance
        weights and the priority write-back use those indices, as `DeviceTD3Learner.update` does."""
        arrays = [self._f32(t) for t in (state, action, reward, next_state, done)]
        b = arrays[0].shape[0]
        if self._arange is None or self._arange.shape[0] < b:
            self._arange = torch.arange(max(b, 1), dtype=torch.int64, device=self.device)
        prio = None
        if self.prioritized and self.replay_buffer.last_batch_inds is not None:
            buf = self.replay_buffer
            prio = (buf.weights, buf.last_batch_inds.to(torch.int64).contiguous(), buf.size)
            buf.last_batch_inds = None
        return self._launch(arrays, self._arange[:b], prio)

    def update_from_buffer(self, batch_size=None):
        """Draw the batch's indices from the replay buffer (`sample_indices`: the same draws as `sample`) and run one
        update that gathers the rows in the kernel."""
        buf = self.replay_buffer
        idx = buf.sample_indices(batch_size or self.cfg.batch_size)
        prio = None
        if self.prioritized:
            prio = (buf.weights, idx, buf.size)
            buf.last_batch_inds = None
        return self._launch((buf.obs, buf.action, buf.reward, buf.next_obs, buf.done), idx, prio)


class FusedTD3Population:
    """K independent TD3 learners (a seed or hyper-parameter sweep, population-based training) updated in ONE launch of K
    thread-block clusters (hk_td3_update_population): member m's update is byte-for-byte the one `FusedTD3Learner` would
    make with the same batch, so the population runs K learners at once on SMs a single learner leaves idle.

    `members[m]` is a full `FusedTD3Learner` whose arena is row m of `arenas` ([K, hk_td3_arena_bytes()] uint8): its
    modules, `state_dict` / `load_state_dict`, `FusedActor.refresh(member.actor)` and a single-member `update` work on
    the live weights.  `configs[m]` is member m's `TD3Config`; every field may differ per member except batch_size,
    buffer_size and prioritized_replay, which the shared `PopulationReplayBuffer` fixes.  Hyper-parameters are read at
    every update, so editing `configs[m]` between calls is PBT's explore step; `copy_member(dst, src)` is its exploit step.

    configs: None (defaults), one TD3Config (copied for each member) or a list of K.  actors / critics: lists of K modules
    or None (fresh ones).  seeds: K target-noise seeds (default 0 .. K-1).  replay_buffer: a PopulationReplayBuffer of
    this K (default: a new one of the configs' buffer_size and prioritized_replay, seed 0)."""

    MAX_K = 64  # HK_TD3_MAX_POPULATION

    def __init__(self, k, configs=None, actors=None, critics=None, seeds=None, replay_buffer=None, device="cuda:0"):
        import ctypes as C
        from . import _lib
        self.k = int(k)
        if not 1 <= self.k <= self.MAX_K:
            raise ValueError(f"FusedTD3Population: k must be in [1, {self.MAX_K}], got {k}")
        self.configs = self._configs(self.k, configs)
        for name, xs in (("actors", actors), ("critics", critics), ("seeds", seeds)):
            if xs is not None and len(xs) != self.k:
                raise ValueError(f"FusedTD3Population: {name} must have k = {self.k} entries, got {len(xs)}")
        cfg0 = self.configs[0]
        if replay_buffer is not None and (replay_buffer.k != self.k or replay_buffer.prioritized != cfg0.prioritized_replay):
            raise ValueError(f"FusedTD3Population: the replay buffer must be a PopulationReplayBuffer of k = {self.k} with "
                             f"prioritized={cfg0.prioritized_replay}")
        from .actor import _cuda_device
        self.device = _cuda_device(device, "FusedTD3Population")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self._C, self._lib = C, _lib
        self.L = _lib.load()
        self.seeds = [int(s) & (2**64 - 1) for s in (seeds if seeds is not None else range(self.k))]
        self.replay_buffer = replay_buffer if replay_buffer is not None else PopulationReplayBuffer(
            self.k, cfg0.buffer_size, device=self.device, prioritized=cfg0.prioritized_replay)
        self.arena_bytes = int(self.L.hk_td3_arena_bytes())
        self.arenas = torch.zeros((self.k, self.arena_bytes), dtype=torch.uint8, device=self.device)
        self.members = [FusedTD3Learner(actor=None if actors is None else actors[m], critic=None if critics is None else critics[m],
                                        config=self.configs[m], device=self.device, seed=self.seeds[m], arena=self.arenas[m])
                        for m in range(self.k)]
        self._scratch, self._scratch_b = None, 0
        self._last_batch = 0
        self.fused_pool = None  # train_population: the FusedActorPool the members act through
        n = self.k
        self._hp = (_lib.TD3HParams * n)()
        self._low, self._range = (C.c_void_p * n)(), (C.c_void_p * n)()
        self._seeds = (C.c_uint64 * n)(*self.seeds)
        self._do_actor = (C.c_uint8 * n)()

    @staticmethod
    def _configs(k, configs):
        if configs is None:
            configs = TD3Config()
        if isinstance(configs, TD3Config):
            configs = [copy.copy(configs) for _ in range(k)]
        configs = list(configs)
        if len(configs) != k:
            raise ValueError(f"FusedTD3Population: configs must have k = {k} entries, got {len(configs)}")
        for f in ("batch_size", "buffer_size", "prioritized_replay"):
            vals = {getattr(c, f) for c in configs}
            if len(vals) != 1:
                raise ValueError(f"FusedTD3Population: {f} must be equal across the members (they share one replay buffer "
                                 f"and one launch), got {sorted(vals)}")
        return configs

    def __len__(self):
        return self.k

    def copy_member(self, dst, src):
        """Make member dst a copy of member src: the whole arena row (weights, targets, Adam moments, step counts and
        noise counter), the critics' action bounds and the actor-step schedule.  configs and seeds stay per member."""
        d, s = self.members[dst], self.members[src]
        self.arenas[dst].copy_(self.arenas[src])
        for net_d, net_s in ((d.critic, s.critic), (d.target_critic, s.target_critic)):
            for k in ("action_low", "action_high", "action_range"):
                getattr(net_d, k).copy_(getattr(net_s, k))
        d.train_step = s.train_step

    def update_from_buffer(self, batch_size=None):
        """One index draw ([K, b] from the population buffer) and one population launch (`update`)."""
        return self.update(self.replay_buffer.sample_indices(batch_size or self.configs[0].batch_size))

    def update(self, idx):
        """One population launch on the batches idx ([K, b] int64 CUDA: global rows of the population buffer, member m's
        inside its own rows; not checked).  Returns ([K] actor losses, NaN for members that made no actor step; [K] critic
        losses) as device tensors; no host sync, graph-capturable."""
        C, lib, buf = self._C, self._lib, self.replay_buffer
        if not (idx.dtype == torch.int64 and idx.dim() == 2 and idx.shape[0] == self.k and idx.is_contiguous()
                and idx.device == self.device):
            raise ValueError(f"FusedTD3Population.update: idx must be a contiguous int64 tensor [{self.k}, b] on {self.device}")
        b = idx.shape[1]
        if not 1 <= b <= FusedTD3Learner.MAX_BATCH:
            raise ValueError(f"FusedTD3Population: batch size must be in [1, {FusedTD3Learner.MAX_BATCH}], got {b}")
        per = int(self.L.hk_td3_scratch_bytes(b))
        if self._scratch is None or self._scratch_b != b:
            self._scratch = torch.empty((self.k, per), dtype=torch.uint8, device=self.device)
            self._scratch_b = b
        for m, mem in enumerate(self.members):
            mem.cfg = self.configs[m]
            mem.train_step += 1
            self._do_actor[m] = int(mem.train_step % mem.cfg.policy_update_freq == 0)
            self._hp[m] = mem._hparams()
            self._low[m], self._range[m] = mem.critic.action_low.data_ptr(), mem.critic.action_range.data_ptr()
        losses = torch.full((self.k, 2), float("nan"), dtype=torch.float32, device=self.device)
        batch = lib.TD3Batch(buf.obs.data_ptr(), buf.action.data_ptr(), buf.reward.data_ptr(), buf.next_obs.data_ptr(),
                             buf.done.data_ptr(), idx.data_ptr())
        if buf.prioritized:
            batch.prio_weights, batch.prio_idx, batch.prio_n = buf.weights.data_ptr(), idx.data_ptr(), buf.size
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            lib.check(self.L.hk_td3_update_population(
                C.c_void_p(self.arenas.data_ptr()), C.c_void_p(self._scratch.data_ptr()), C.byref(batch), b, self.k, self._hp,
                self._low, self._range, self._seeds, self._do_actor, C.c_void_p(losses.data_ptr()), self.device.index,
                C.c_void_p(stream)))
        self._last_batch = b
        self.last_do_actor = [bool(v) for v in self._do_actor]
        return losses[:, 0], losses[:, 1]

    def last_importance_weights(self):
        """[K, B] importance weights of the last update (ones for uniform batches), computed in the kernel."""
        return self._scratch.view(torch.float32)[:, :self._last_batch]

    def refresh_pool(self, pool):
        """Repack slots 0 .. K-1 of `pool` (a FusedActorPool) from the members' live actors in one hk_actor_pack_many
        launch (no host sync); other slots are not touched."""
        C = self._C
        if len(pool) < self.k or pool.device != self.device:
            raise ValueError(f"refresh_pool needs a FusedActorPool of >= {self.k} slots on {self.device}")
        with torch.cuda.device(self.device):
            self._lib.check(self.L.hk_actor_pack_many(
                C.c_void_p(self.arenas.data_ptr()), self.arena_bytes // 4, self.k, C.c_void_p(pool.table.data_ptr()),
                self.device.index, C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)))
        return pool


@torch.no_grad()
def _explore(actor, obs, noise_scale, gen):
    a = actor(obs)
    return (a + torch.randn(a.shape, device=a.device, generator=gen) * noise_scale).clamp(-1, 1)


def train(env_or_pool, learner, ticks, updates_per_tick=1, noise_scale=None, warmup_ticks=8, fused=False, noise=None):
    """Batched form of TD3Trainer's loop (rl/training/train.py:135-172): every tick all envs act with Gaussian
    exploration noise, their transitions (terminal observation as next_obs on done) go to the learner's device replay
    buffer, and `updates_per_tick` learner steps follow.  Returns the mean critic loss of the last tick (device scalar).

    fused=True: the envs act through `learner.fused_actor`, a `FusedActor` mirror of `learner.actor` (created on first
    use, seeded with the learner's seed), with the exploration noise drawn in the kernel: one launch per tick.  The
    mirror is repacked on the device (`FusedActor.refresh`: no host sync) at the start of the call and after every tick
    whose updates changed the actor, so every tick acts with the current weights.  The learner itself still trains the
    fp32 module; only the behaviour policy runs in bf16 / TF32 (TD3 is off-policy).

    noise: an `ExplorationNoise` of N rows (fused=True only, instead of noise_scale): the envs explore with its slot 0
    (e.g. Ornstein-Uhlenbeck noise), each tick passes the previous tick's done as `reset`, and the rows whose episode
    ended on the last tick are zeroed before returning, so every episode starts from a zero noise state, across calls
    too.  `noise.set(0, sigma=...)` between calls anneals it."""
    from .actor import FusedActor
    from .training import OpponentPool
    if noise is not None:
        if noise_scale is not None:
            raise ValueError("train: pass either noise_scale= or noise=, not both")
        if not fused:
            raise ValueError("train: noise=ExplorationNoise needs fused=True (its state exists only in the fused launch)")
    pool = env_or_pool if isinstance(env_or_pool, OpponentPool) else None
    env = pool.env if pool else env_or_pool
    buf = learner.replay_buffer
    scale = learner.cfg.action_noise_scale if noise_scale is None else noise_scale
    mirror = None
    if fused:
        if learner.fused_actor is None:
            learner.fused_actor = FusedActor(learner.actor, device=learner.device, seed=learner.seed)
        mirror = learner.fused_actor.refresh(learner.actor)
    obs = env.obs.clone()
    loss = done = None
    for t in range(ticks):
        if noise is not None:
            a = mirror(obs, noise=noise, reset=done)
        elif mirror is not None:
            a = mirror(obs, noise=scale)
        else:
            a = _explore(learner.actor, obs, scale, learner.gen)
        nobs, reward, done, _, _ = pool.step(a) if pool else env.step(a.contiguous())
        nxt = torch.where(done.to(torch.bool).unsqueeze(1), env.final_obs, nobs) if env.final_obs is not None else nobs
        buf.push(obs, a, reward, nxt, done)
        obs = nobs.clone()
        if t >= warmup_ticks:
            changed = False
            for _ in range(updates_per_tick):
                actor_loss, loss = learner.update_from_buffer()
                changed |= actor_loss is not None
            if changed and mirror is not None:
                mirror.refresh(learner.actor)
    if noise is not None and done is not None:
        noise.reset(done)  # episodes that ended on the last tick start the next call from x = 0
    return loss


def train_population(env_or_pool, population, ticks, updates_per_tick=1, noise_scale=None, warmup_ticks=8, noise=None):
    """`train(..., fused=True)` for a `FusedTD3Population`: the env's N rows are split into K equal contiguous blocks, and
    block m acts through member m -- one noisy `FusedActorPool` launch per tick with the constant choice row // (N / K),
    exploration noise keyed on the global row.  The transitions go to the population's buffer (block m to member m),
    `updates_per_tick` population launches follow each tick after `warmup_ticks`, and after a tick whose updates stepped
    any actor one hk_actor_pack_many launch repacks all K slots.  Without `noise=`, the exploration sigma is one scalar for the
    population (noise_scale, or the members' action_noise_scale, which must then be equal).  An `OpponentPool` works as with
    `train` (player-1 columns only).  Returns the [K] critic losses of the last update (device tensor; None if none ran).

    noise: an `ExplorationNoise` of N rows and K slots (instead of noise_scale): block m explores with slot m, so the
    members may explore differently (their action_noise_scale is then not consulted), and each tick passes the previous
    tick's done as `reset` (rows whose episode ended on the last tick are zeroed before returning, as in `train`).
    `noise.set(m, ...)` changes member m's exploration (a PBT explore step) between calls."""
    from .actor import FusedActorPool
    from .training import OpponentPool
    pool = env_or_pool if isinstance(env_or_pool, OpponentPool) else None
    env = pool.env if pool else env_or_pool
    k, n = population.k, env.num_envs
    if n % k:
        raise ValueError(f"train_population: {n} envs do not split into {k} equal blocks")
    if noise is not None:
        if noise_scale is not None:
            raise ValueError("train_population: pass either noise_scale= or noise=, not both")
        if noise.slots != k or noise.n != n:
            raise ValueError(f"train_population: noise= needs an ExplorationNoise of {n} rows and {k} slots (one per member), "
                             f"got {noise.n} rows and {noise.slots} slots")
    elif noise_scale is None:
        scales = {c.action_noise_scale for c in population.configs}
        if len(scales) != 1:
            raise ValueError(f"train_population: the members' action_noise_scale differ ({sorted(scales)}); the pooled actor "
                             f"launch takes one sigma, so pass noise_scale=")
        noise_scale = scales.pop()
    buf = population.replay_buffer
    if population.fused_pool is None:
        population.fused_pool = FusedActorPool([m.actor for m in population.members], device=population.device,
                                               seed=population.seeds[0])
    acting = population.refresh_pool(population.fused_pool)
    choice = (torch.arange(n, device=env.device) // (n // k)).to(torch.int32)
    obs = env.obs.clone()
    loss = done = None
    for t in range(ticks):
        if noise is not None:
            a = acting(obs, choice, noise=noise, reset=done)
        else:
            a = acting(obs, choice, noise=noise_scale)
        nobs, reward, done, _, _ = pool.step(a) if pool else env.step(a.contiguous())
        nxt = torch.where(done.to(torch.bool).unsqueeze(1), env.final_obs, nobs) if env.final_obs is not None else nobs
        buf.push(obs, a, reward, nxt, done)
        obs = nobs.clone()
        if t >= warmup_ticks:
            changed = False
            for _ in range(updates_per_tick):
                _, loss = population.update_from_buffer()
                changed |= any(population.last_do_actor)
            if changed:
                population.refresh_pool(acting)
    if noise is not None and done is not None:
        noise.reset(done)  # episodes that ended on the last tick start the next call from x = 0
    return loss
