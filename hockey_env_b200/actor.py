"""On-device policy plumbing for BASELINE config 5 (self-play rollout with a TD3 actor) -- SURVEY.md section 8f rank 2.

The actor is the reference's `ActorNetwork` (rl/td3/networks.py:6-20: 18 -> 256 -> 256 -> 4, tanh after every layer);
it consumes the env's observation tensor in place (no host round trip) and its output feeds `HockeyVecEnv.step`.
The dense layers are plain library matmuls (torch/cuBLAS): they are the op adjacent to the hot path, not the path.
"""
import torch
from torch import nn


class ActorNetwork(nn.Module):
    def __init__(self, obs_dim=18, action_dim=4, hidden=256):
        super().__init__()
        self.fc1 = nn.Linear(obs_dim, hidden)
        self.fc2 = nn.Linear(hidden, hidden)
        self.fc3 = nn.Linear(hidden, action_dim)

    def forward(self, obs):
        x = torch.tanh(self.fc1(obs))
        x = torch.tanh(self.fc2(x))
        return torch.tanh(self.fc3(x))


def load_td3_actor(path, device="cuda:0", name=None):
    """The reference's trained policy as an on-device module.  `path` is either a reference checkpoint written by
    `TD3Agent.save` (rl/td3/agent.py:269-275: a dict whose `policy` entry is the ActorNetwork state_dict) or an
    `.npz` of float32 arrays `<name>.fc1.weight` ... `<name>.fc3.bias` (tests/golden/td3_actors.npz, extracted from
    those checkpoints by tests/golden/make_actor_fixtures.py)."""
    if str(path).endswith(".npz"):
        import numpy as np
        z = np.load(path)
        names = sorted({k.split(".")[0] for k in z.files})
        if name is None:
            if len(names) != 1:
                raise ValueError(f"{path} holds several actors {names}: pass name=")
            name = names[0]
        if name not in names:
            raise ValueError(f"no actor {name!r} in {path}; have {names}")
        sd = {k[len(name) + 1:]: torch.from_numpy(z[k]) for k in z.files if k.startswith(name + ".")}
    else:
        ckpt = torch.load(path, map_location="cpu", weights_only=False)
        sd = ckpt["policy"] if "policy" in ckpt else ckpt
    hidden, obs_dim = sd["fc1.weight"].shape
    actor = ActorNetwork(obs_dim=obs_dim, action_dim=sd["fc3.weight"].shape[0], hidden=hidden)
    actor.load_state_dict(sd)
    return actor.to(device).eval()


def _cuda_device(device, who):
    from . import _lib
    device = torch.device(device)
    if device.type != "cuda" or not torch.cuda.is_available():
        raise _lib.HockeyLibraryError(f"{who} needs a CUDA device: the actor kernel has no CPU fallback")
    return device


_PARAM_SHAPES = (("fc1.weight", (256, 18)), ("fc1.bias", (256,)), ("fc2.weight", (256, 256)), ("fc2.bias", (256,)),
                 ("fc3.weight", (4, 256)), ("fc3.bias", (4,)))


def _live_params(actor, device, who):
    """The module's six parameter tensors on `device` as contiguous fp32 (in place when they already are: no copy, no
    host sync), in hk_actor_pack's order w1, b1, w2, b2, w3, b3."""
    sd = actor.state_dict(keep_vars=True)
    out = []
    for name, shape in _PARAM_SHAPES:
        t = sd[name].detach()
        if tuple(t.shape) != shape:
            raise ValueError(f"{who} implements the reference architecture 18 -> 256 -> 256 -> 4")
        if t.device.type != "cuda" or (t.device.index or 0) != (device.index or 0):
            raise ValueError(f"{who}: the module's parameters are on {t.device}, the packed block on {device}")
        out.append(t.to(torch.float32).contiguous())
    return out


def _pack_on_device(L, lib, actor, dst, device, who):
    """hk_actor_pack of `actor`'s live parameters into the 16-byte aligned block at `dst` (a uint8 CUDA tensor view)."""
    import ctypes as C
    ps = _live_params(actor, device, who)
    with torch.cuda.device(device):
        lib.check(L.hk_actor_pack(*[C.c_void_p(p.data_ptr()) for p in ps], C.c_void_p(dst.data_ptr()), device.index or 0,
                                  C.c_void_p(torch.cuda.current_stream(device).cuda_stream)))


def _noise_args(noise, noise_clip):
    sigma = float(noise)
    if not (sigma >= 0.0 and sigma != float("inf")):
        raise ValueError("noise must be a finite standard deviation >= 0")
    clip = 0.0 if noise_clip is None else float(noise_clip)
    if clip != clip:
        raise ValueError("noise_clip must not be NaN")
    return sigma, clip


def _reference_state_dict(actor, who):
    """The fp32 CPU state dict of an ActorNetwork-shaped module, checked against the reference architecture."""
    sd = {k: v.detach().to("cpu", torch.float32) for k, v in actor.state_dict().items()}
    if tuple(sd["fc1.weight"].shape) != (256, 18) or tuple(sd["fc2.weight"].shape) != (256, 256) or tuple(sd["fc3.weight"].shape) != (4, 256):
        raise ValueError(f"{who} implements the reference architecture 18 -> 256 -> 256 -> 4")
    return sd


class FusedActor:
    """The same network as ONE fused sm_100a tensor-core kernel (csrc/hk_actor.cuh, hk_actor_forward): weights resident in
    shared memory (layer 1 TF32, layers 2-3 bf16), fp32 accumulation in tensor memory, hidden activations never leave the SM.  Callable like the
    module: obs [N,18] float32 CUDA tensor -> actions [N,4] (a persistent output buffer, overwritten by the next call;
    pass `out=` to write into columns 0..3 of an existing [N,4] / [N,8] action tensor).  There is no fallback: without the
    CUDA library or a GPU this raises.

    For a policy that is being trained: `refresh(module)` repacks the block on the device from the module's live
    parameters (hk_actor_pack: no CPU copy, no host sync, graph-capturable), and `noise=sigma` adds TD3 exploration
    noise in the kernel's epilogue, clamp(actor(obs) + clip(sigma * z, +-noise_clip), -1, 1) with z drawn by Philox from
    (seed, row0 + row, counter).  The counter is a device int64 (`self.counter`) that every noisy call advances, so
    consecutive calls -- and the replays of a captured graph -- draw fresh noise."""

    PARAM_BYTES = 256 * 24 * 4 + 256 * 256 * 2 + 16 * 256 * 2 + 2 * 256 * 4 + 16 * 4  # hk_actor_param_bytes()

    def __init__(self, actor, device="cuda:0", seed=0):
        import ctypes as C
        from . import _lib
        self._C, self._lib = C, _lib
        self.L = _lib.load()
        self.device = _cuda_device(device, "FusedActor")
        self.params = self.pack(_reference_state_dict(actor, "FusedActor")).to(self.device)
        assert self.params.numel() == int(self.L.hk_actor_param_bytes())
        self._out = None
        self.seed = int(seed) & (2**64 - 1)
        self.counter = torch.zeros(1, dtype=torch.int64, device=self.device)

    def refresh(self, actor):
        """Repack the block in place from `actor`'s live parameters (fp32 tensors on this device), on the current
        stream: no CPU copy, no host sync.  The result equals `FusedActor.pack` of the same weights byte for byte."""
        _pack_on_device(self.L, self._lib, actor, self.params, self.device, "FusedActor.refresh")
        return self

    @staticmethod
    def _core_matrix_order(w, n_pad, k_pad, dtype):
        """[N, K] float weight -> bytes in UMMA K-major core-matrix order (8-row x 16-byte core matrices, no swizzle):
        with e = 16 / itemsize elements per 16-byte chunk, element (n, k) sits at
        (k // e) * (n_pad * 16) + n * 16 + (k % e) * itemsize bytes.  dtype bfloat16, or float32 for the TF32 layer."""
        full = torch.zeros((n_pad, k_pad), dtype=torch.float32)
        full[:w.shape[0], :w.shape[1]] = w
        e = 16 // torch.empty((), dtype=dtype).element_size()
        return full.to(dtype).view(n_pad, k_pad // e, e).permute(1, 0, 2).contiguous().view(torch.uint8).flatten()

    @classmethod
    def pack(cls, sd):
        b3 = torch.zeros(16, dtype=torch.float32)
        b3[:4] = sd["fc3.bias"]
        parts = [cls._core_matrix_order(sd["fc1.weight"], 256, 24, torch.float32),
                 cls._core_matrix_order(sd["fc2.weight"], 256, 256, torch.bfloat16),
                 cls._core_matrix_order(sd["fc3.weight"], 16, 256, torch.bfloat16),
                 sd["fc1.bias"].contiguous().view(torch.uint8).flatten(),
                 sd["fc2.bias"].contiguous().view(torch.uint8).flatten(), b3.view(torch.uint8).flatten()]
        return torch.cat(parts).contiguous()

    def __call__(self, obs, out=None, noise=0.0, noise_clip=None, row0=0):
        """actions = actor(obs); with noise > 0, clamp(actor(obs) + clip(noise * z, +-noise_clip), -1, 1) (noise_clip None
        or <= 0: no clip), then the counter advances.  `row0` is the global index of row 0 (shards of one batch pass
        their offset to draw the same noise as one call over the whole batch)."""
        if not (obs.is_cuda and obs.dtype == torch.float32 and obs.is_contiguous() and obs.dim() == 2 and obs.shape[1] == 18):
            raise ValueError("FusedActor expects a contiguous float32 CUDA tensor [N, 18]")
        sigma, clip = _noise_args(noise, noise_clip)
        n = obs.shape[0]
        if out is None:
            if self._out is None or self._out.shape[0] != n:
                self._out = torch.empty((n, 4), dtype=torch.float32, device=obs.device)
            out = self._out
        if not (out.is_cuda and out.dtype == torch.float32 and out.dim() == 2 and out.shape[0] == n and out.stride(1) == 1 and out.shape[1] >= 4):
            raise ValueError("out must be a float32 CUDA tensor [N, >= 4] with unit column stride")
        C = self._C
        with torch.cuda.device(obs.device):
            stream = C.c_void_p(torch.cuda.current_stream(obs.device).cuda_stream)
            if sigma == 0.0:
                self._lib.check(self.L.hk_actor_forward(C.c_void_p(self.params.data_ptr()), C.c_void_p(obs.data_ptr()),
                                                        C.c_void_p(out.data_ptr()), int(out.stride(0)), n, obs.device.index or 0, stream))
            else:
                self._lib.check(self.L.hk_actor_forward_noisy(
                    C.c_void_p(self.params.data_ptr()), C.c_void_p(obs.data_ptr()), C.c_void_p(out.data_ptr()), int(out.stride(0)), n,
                    self.seed, C.c_void_p(self.counter.data_ptr()), sigma, clip, int(row0), obs.device.index or 0, stream))
                self.counter.add_(1)
        return out[:, :4] if out.shape[1] != 4 else out


class FusedActorPool:
    """K frozen actors (self-play snapshots, a league) evaluated per row in ONE tensor-core pass
    (csrc/hk_actor.cuh k_actor_pool_mlp, hk_actor_forward_pool): row i goes through snapshot choice[i].  The rows are
    grouped by snapshot on the device (no host sync; graph-capturable), and each written row equals
    `FusedActor(snapshot choice[i])(obs)[i]` bit for bit.  The table is one [K, hk_actor_param_bytes()] uint8 device
    tensor of `FusedActor.pack` blocks; `add` appends one (and re-allocates the table: re-capture graphs after it), `set`
    repacks one slot in place on the device.  `noise=` / `noise_clip=` add the epilogue noise of `FusedActor` (keyed on
    the row, not on the snapshot).  There is no fallback: without the CUDA library or a GPU this raises."""

    MAX_K = 4096

    def __init__(self, actors=(), device="cuda:0", seed=0):
        import ctypes as C
        from . import _lib
        self._C, self._lib = C, _lib
        self.L = _lib.load()
        self.device = _cuda_device(device, "FusedActorPool")
        self.table = self.pack(actors).to(self.device)
        self._out = None
        self._scratch = torch.empty(0, dtype=torch.uint8, device=self.device)
        self.seed = int(seed) & (2**64 - 1)
        self.counter = torch.zeros(1, dtype=torch.int64, device=self.device)

    @staticmethod
    def pack(actors):
        """[K, param_bytes] uint8 (CPU): block s is `FusedActor.pack` of actors[s], at byte offset s * param_bytes of
        the flattened table."""
        blocks = [FusedActor.pack(_reference_state_dict(a, "FusedActorPool")) for a in actors]
        return torch.stack(blocks) if blocks else torch.empty((0, FusedActor.PARAM_BYTES), dtype=torch.uint8)

    def __len__(self):
        return self.table.shape[0]

    def add(self, actor):
        """Append one snapshot; returns its index (the choice value that selects it)."""
        if len(self) >= self.MAX_K:
            raise ValueError(f"FusedActorPool holds at most {self.MAX_K} snapshots")
        blk = self.pack([actor]).to(self.device)
        self.table = torch.cat([self.table, blk])
        return len(self) - 1

    def set(self, i, actor):
        """Repack slot `i` in place from `actor`'s live parameters (hk_actor_pack into the table: no CPU copy, no host
        sync); the other slots are not touched."""
        i = int(i)
        if not 0 <= i < len(self):
            raise IndexError(f"FusedActorPool slot {i} out of range [0, {len(self)})")
        _pack_on_device(self.L, self._lib, actor, self.table[i], self.device, "FusedActorPool.set")

    def __call__(self, obs, choice, out=None, noise=0.0, noise_clip=None, row0=0):
        """obs [N,18] float32 CUDA, choice int32 / int64 CUDA [N] -> act[i] = actor_{choice[i]}(obs[i]) for choice[i] in
        [0, K); other rows are not written.  out=None: a persistent [N,4] buffer (overwritten by the next call) whose
        skipped rows are 0; or pass `out` = an [N, >= 4] float32 view with unit column stride (e.g. `a8[:, 4:]` of the
        [N,8] action tensor): columns 0..3 of its written rows change, nothing else.  noise / noise_clip / row0 as for
        `FusedActor`; a noisy call advances the counter."""
        if not (obs.is_cuda and obs.dtype == torch.float32 and obs.is_contiguous() and obs.dim() == 2 and obs.shape[1] == 18):
            raise ValueError("FusedActorPool expects a contiguous float32 CUDA tensor [N, 18]")
        sigma, clip = _noise_args(noise, noise_clip)
        n, k = obs.shape[0], len(self)
        if k == 0:
            raise ValueError("FusedActorPool is empty: add() a snapshot first")
        if not (isinstance(choice, torch.Tensor) and choice.is_cuda and choice.dtype in (torch.int32, torch.int64)
                and choice.shape == (n,) and choice.device == obs.device == self.table.device):
            raise ValueError("choice must be an int32 or int64 CUDA tensor [N], on the pool's device like obs")
        if choice.dtype == torch.int64:  # out-of-range values stay out of range after the narrowing
            choice = torch.where((choice >= 0) & (choice < k), choice, -1).to(torch.int32)
        choice = choice.contiguous()
        if out is None:
            if self._out is None or self._out.shape[0] != n or self._out.device != obs.device:
                self._out = torch.empty((n, 4), dtype=torch.float32, device=obs.device)
            out = self._out
            out.zero_()
        if not (out.is_cuda and out.dtype == torch.float32 and out.dim() == 2 and out.shape[0] == n and out.stride(1) == 1 and out.shape[1] >= 4):
            raise ValueError("out must be a float32 CUDA tensor [N, >= 4] with unit column stride")
        if n == 0:
            return out[:, :4]
        need = int(self.L.hk_actor_pool_scratch_bytes(n, k))
        if need < 0:
            self._lib.check(need)
        if self._scratch.numel() < need:
            self._scratch = torch.empty(need, dtype=torch.uint8, device=self.device)
        C = self._C
        with torch.cuda.device(obs.device):
            stream = C.c_void_p(torch.cuda.current_stream(obs.device).cuda_stream)
            if sigma == 0.0:
                self._lib.check(self.L.hk_actor_forward_pool(C.c_void_p(self.table.data_ptr()), k, C.c_void_p(choice.data_ptr()),
                                                             C.c_void_p(obs.data_ptr()), C.c_void_p(out.data_ptr()), int(out.stride(0)),
                                                             n, C.c_void_p(self._scratch.data_ptr()), obs.device.index or 0, stream))
            else:
                self._lib.check(self.L.hk_actor_forward_pool_noisy(
                    C.c_void_p(self.table.data_ptr()), k, C.c_void_p(choice.data_ptr()), C.c_void_p(obs.data_ptr()),
                    C.c_void_p(out.data_ptr()), int(out.stride(0)), n, C.c_void_p(self._scratch.data_ptr()), self.seed,
                    C.c_void_p(self.counter.data_ptr()), sigma, clip, int(row0), obs.device.index or 0, stream))
                self.counter.add_(1)
        return out[:, :4] if out.shape[1] != 4 else out


@torch.no_grad()
def actor_rollout(env, actor, steps, opponent_actor=None):
    """`steps` ticks of `env` (a HockeyVecEnv with p1 external) driven by `actor`; player 2 is the env's in-kernel
    BasicOpponent, or `opponent_actor` acting on obs_agent_two() (the PolicyOpponent pattern, hockey_env.py:908-922)
    when the env was built with p2=None.  Returns the env's episode statistics."""
    obs = env.obs
    for _ in range(steps):
        a1 = actor(obs)
        if opponent_actor is not None:
            a2 = opponent_actor(env.obs_agent_two())
            obs, *_ = env.step(torch.cat([a1, a2], dim=1).contiguous())
        else:
            obs, *_ = env.step(a1.contiguous())
    return env.stats()
