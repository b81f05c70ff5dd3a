"""Host-side mirror of the reference's gym-facing surface (hockey/hockey_env.py) over the CUDA library.

`HockeyVecEnv` is the batched, zero-copy API (torch CUDA tensors in/out, one kernel launch per tick).
`HockeyEnv`, `HockeyEnv_BasicOpponent`, `BasicOpponent`, `PolicyOpponent`, `Mode` keep the reference's
names, signatures and semantics (single env = batch of 1) so that code written against
`hockey.hockey_env` runs unchanged.  PyTorch is used only for device memory and streams.
"""
import ctypes as C
import math
from enum import Enum

import numpy as np
import torch

from . import _lib

# constants of the reference module (hockey_env.py:17-37)
FPS = 50
SCALE = 60.0
VIEWPORT_W = 600
VIEWPORT_H = 480
W = VIEWPORT_W / SCALE
H = VIEWPORT_H / SCALE
CENTER_X = W / 2
CENTER_Y = H / 2
ZONE = W / 20
MAX_ANGLE = math.pi / 3
MAX_TIME_KEEP_PUCK = 15
GOAL_SIZE = 75
RACKETPOLY = [(-10, 20), (+5, 20), (+5, -20), (-10, -20), (-18, -10), (-21, 0), (-18, 10)]
RACKETFACTOR = 1.2
FORCEMULTIPLIER = 6000
SHOOTFORCEMULTIPLIER = 60
TORQUEMULTIPLIER = 400
MAX_PUCK_SPEED = 25


class Mode(Enum):  # hockey_env.py:78-81
    NORMAL = 0
    TRAIN_SHOOTING = 1
    TRAIN_DEFENSE = 2


def _as_mode(value):
    """Accept an Enum member, a name or an int, with the reference's errors (hockey_env.py:758-779)."""
    if isinstance(value, Mode):
        return value
    if isinstance(value, str):
        try:
            return Mode[value]
        except KeyError:
            raise ValueError(f"{value} is not a valid name for {Mode.__name__}")
    if isinstance(value, (int, np.integer)) and not isinstance(value, bool):
        try:
            return Mode(int(value))
        except ValueError:
            raise ValueError(f"{value} is not a valid value for {Mode.__name__}")
    raise TypeError("Input value must be an Enum, name (str), or value (int)")


_POLICY_IDS = {
    None: _lib.POLICY_EXTERNAL, "external": _lib.POLICY_EXTERNAL,
    "weak": _lib.POLICY_BASIC_WEAK, "basic_weak": _lib.POLICY_BASIC_WEAK,
    "strong": _lib.POLICY_BASIC_STRONG, "basic_strong": _lib.POLICY_BASIC_STRONG,
    "random": _lib.POLICY_RANDOM, "zero": _lib.POLICY_ZERO,
    "per_env": _lib.POLICY_PER_ENV,  # player 2 only: one code per env (HockeyVecEnv.set_opponent_policies)
}


def _policy_id(p):
    if isinstance(p, (int, np.integer)) and not isinstance(p, bool):
        return int(p)
    try:
        return _POLICY_IDS[p]
    except KeyError:
        raise ValueError(f"unknown policy {p!r}; use one of {sorted(k for k in _POLICY_IDS if k)}")


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


class HockeyVecEnv:
    """N independent HockeyEnvs stepped by one CUDA launch per tick.

    All tensors returned by `reset`/`step` are persistent device buffers owned by this object and are
    overwritten by the next call (zero-copy; clone() to keep).  Work is enqueued on the current torch
    CUDA stream; nothing synchronises the host.

    p1 / p2: None (actions come from the caller) or 'weak' / 'strong' (in-kernel BasicOpponent,
    hockey_env.py:781-833) / 'random' / 'zero'.  With p2 set, `step` takes [N,4] actions like
    HockeyEnv_BasicOpponent (hockey_env.py:875-886); otherwise [N,8] like HockeyEnv.
    p2='per_env': every env has its own opponent code (`set_opponent_policies`), the batched form of drawing an
    opponent per episode from a pool (rl/training/opponent_manager.py:62-91); `step` then takes [N,8] actions whose
    columns 4..7 are only read by the envs whose code is 'external' (e.g. a self-play snapshot's output).

    mode: one Mode (or name / int) for every env, or one per env (a sequence or a uint8 tensor [N]).  Per-env modes are
    the batched form of the reference's `mode` setter: the handle is created, the modes are set as reset codes
    (`set_reset_modes`) and every env is reset once with one_starting=True, so that this reset starts each env's
    episode 1 (episode 0 is the creation's own reset, hockey_env.py:155).  Every later reset -- `reset` or an
    auto-reset -- starts the next episode in the mode `reset_modes` holds for the env; `modes()` gives the mode each
    env plays now.
    """

    def __init__(self, num_envs, mode=Mode.NORMAL, keep_mode=True, device="cuda:0", seed=0, env_id_offset=0,
                 auto_reset=True, p1=None, p2=None, want_agent_two=False):
        self.L = _lib.load()
        if not torch.cuda.is_available():
            raise _lib.HockeyLibraryError("no CUDA device: hockey_env_b200 has no CPU fallback")
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise ValueError("HockeyVecEnv needs a CUDA device")
        self.num_envs = int(num_envs)
        per_env_modes = None
        if isinstance(mode, torch.Tensor) or (isinstance(mode, (list, tuple, np.ndarray)) and np.ndim(mode) == 1):
            per_env_modes = mode
            mode = Mode.NORMAL  # the creation mode: record word HK_S_MODE = 0 stands for it
        self._mode = _as_mode(mode)
        self.keep_mode = bool(keep_mode)
        self.auto_reset = bool(auto_reset)
        self.p1 = _policy_id(p1)
        self.p2 = _policy_id(p2)
        if self.p1 == _lib.POLICY_PER_ENV:
            raise ValueError("'per_env' is a player-2 policy")
        self.opponent_codes = None
        self.reset_modes = None
        self.want_agent_two = bool(want_agent_two)
        dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        h = C.c_void_p()
        _lib.check(self.L.hk_create(C.byref(h), self.num_envs, self._mode.value, int(self.keep_mode), dev_index,
                                    int(seed) & 0xFFFFFFFFFFFFFFFF, int(env_id_offset)))
        self._h = h
        n, d = self.num_envs, self.device
        self.obs = torch.empty((n, 18), dtype=torch.float32, device=d)
        self.reward = torch.empty(n, dtype=torch.float32, device=d)
        self.done = torch.empty(n, dtype=torch.uint8, device=d)
        self.truncated = torch.zeros(n, dtype=torch.bool, device=d)  # always False (hockey_env.py:695)
        self.info = torch.empty((n, 4), dtype=torch.float32, device=d)
        self.final_obs = torch.empty((n, 18), dtype=torch.float32, device=d) if self.auto_reset else None
        self.obs2 = self.reward2 = self.info2 = None
        if self.want_agent_two:
            self.obs2 = torch.empty((n, 18), dtype=torch.float32, device=d)
            self.reward2 = torch.empty(n, dtype=torch.float32, device=d)
            self.info2 = torch.empty((n, 4), dtype=torch.float32, device=d)
        with torch.cuda.device(self.device):
            _lib.check(self.L.hk_get_obs(self._h, _ptr(self.obs), _ptr(self.obs2), self._stream()))
        if self.p2 == _lib.POLICY_PER_ENV:
            self.set_opponent_policies(torch.full((n,), _lib.POLICY_BASIC_WEAK, dtype=torch.uint8, device=d))
        self._modes = torch.empty(n, dtype=torch.uint8, device=d)
        if per_env_modes is not None:
            self.set_reset_modes(per_env_modes)
            self.reset(one_starting=True)

    def set_opponent_policies(self, codes):
        """Per-env player-2 policy codes: uint8 CUDA tensor [N] of 0 external / 1 weak / 2 strong / 3 random / 4 zero
        (or a list of policy names).  The tensor is kept and read by every step; rewrite `env.opponent_codes` in place
        (e.g. `codes[done.bool()] = new`) to re-draw opponents for finished episodes without a host round trip."""
        if not isinstance(codes, torch.Tensor):
            codes = torch.tensor([_policy_id(c) for c in codes], dtype=torch.uint8)
        codes = codes.to(device=self.device, dtype=torch.uint8).contiguous()
        if codes.shape != (self.num_envs,):
            raise ValueError("codes must be [num_envs]")
        with torch.cuda.device(self.device):
            torch.cuda.current_stream(self.device).synchronize()
            _lib.check(self.L.hk_set_opponent_policies(self._h, _ptr(codes)))
        self.opponent_codes = codes
        return codes

    def _mode_codes(self, modes, name):
        """A scalar mode (Mode / name / int) broadcast to [N], or N of them, as a uint8 device tensor."""
        if isinstance(modes, torch.Tensor):
            return self._per_env(modes, torch.uint8, name)
        if isinstance(modes, (list, tuple, np.ndarray)) and np.ndim(modes) == 1:
            return self._per_env(np.array([_as_mode(m).value for m in modes], dtype=np.uint8), torch.uint8, name)
        return self._per_env(_as_mode(modes).value, torch.uint8, name)

    def set_reset_modes(self, modes):
        """Mode of the episode every later reset of an env starts (explicit `reset` or auto-reset): one Mode for all,
        a sequence of N, or a uint8 CUDA tensor [N] of 0 NORMAL / 1 TRAIN_SHOOTING / 2 TRAIN_DEFENSE.  The tensor is kept
        as `env.reset_modes` and read by every reset; rewrite it in place (e.g. `env.reset_modes[done.bool()] = m`) to
        move envs between modes per episode without a host round trip.  None clears it: every env keeps its mode."""
        codes = None if modes is None else self._mode_codes(modes, "modes")
        with torch.cuda.device(self.device):
            torch.cuda.current_stream(self.device).synchronize()  # the library validates the codes on the default stream
            _lib.check(self.L.hk_set_reset_modes(self._h, _ptr(codes)))
        self.reset_modes = codes
        return codes

    def modes(self):
        """uint8 [N] device tensor: the mode of each env's running episode (a persistent buffer, overwritten by the next
        call; asynchronous like `step`)."""
        with torch.cuda.device(self.device):
            _lib.check(self.L.hk_get_modes(self._h, _ptr(self._modes), self._stream()))
        return self._modes

    @property
    def max_timesteps(self):
        """250 (NORMAL) or 80 while every env plays the constructor's mode; None once envs may play other modes
        (reset codes are set): see `modes()`."""
        if self.reset_modes is not None:
            return None
        return 250 if self._mode == Mode.NORMAL else 80

    # -- plumbing ---------------------------------------------------------------------------------
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def close(self):
        if getattr(self, "_h", None):
            self.L.hk_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def mode(self):
        """The constructor's mode while every env plays it; None once envs may play other modes (see `modes()`)."""
        return None if self.reset_modes is not None else self._mode

    @property
    def action_dim(self):
        ext = (self.p1 == _lib.POLICY_EXTERNAL) + (self.p2 == _lib.POLICY_EXTERNAL)
        return 4 * ext

    def _info_dict(self, info):
        return {"winner": info[:, 0], "reward_closeness_to_puck": info[:, 1], "reward_touch_puck": info[:, 2],
                "reward_puck_direction": info[:, 3]}

    # -- reference surface, batched ------------------------------------------------------------------
    def _per_env(self, value, dtype, name):
        """A scalar (python or numpy, also 0-d) broadcast to [N], or a [N] array/tensor, as a contiguous device tensor."""
        if isinstance(value, torch.Tensor):
            t = value
        else:
            t = torch.as_tensor(np.asarray(value))
        if t.dim() == 0:
            return torch.full((self.num_envs,), t.item(), dtype=dtype, device=self.device)
        if tuple(t.shape) != (self.num_envs,):
            raise ValueError(f"{name} must be a scalar or have shape ({self.num_envs},), got {tuple(t.shape)}")
        return t.to(device=self.device, dtype=dtype).contiguous()

    def reset(self, mask=None, one_starting=None, seed=None, mode=None):
        """HockeyEnv.reset (hockey_env.py:345-418) for the envs selected by `mask` (bool/uint8 [N], None = all).
        one_starting: None = alternate like the reference, a bool, or an int8 array/tensor [N] (1 / 0 / -1 = alternate).
        seed: None = every env continues its own random stream; an int s = env i is reset with seed s + i (the
        gymnasium vector convention); an int64 array/tensor [N] = one seed per env (negative = own stream).  A seeded
        reset draws from that seed alone, like the reference's reseeding (hockey_env.py:347): same seed, same start.
        mode: None = the mode `reset_modes` holds (or keep), a Mode for all or N of them = the reference's
        reset(mode=...): the reset envs' codes in `reset_modes` are rewritten first, so that their later auto-resets
        keep that mode too."""
        m = None
        if mask is not None:
            m = self._per_env(mask, torch.uint8, "mask")
        if mode is not None:
            codes = self._mode_codes(mode, "mode")
            if self.reset_modes is None:
                self.set_reset_modes(self.modes().clone())
            if m is None:
                self.reset_modes.copy_(codes)
            else:
                self.reset_modes.copy_(torch.where(m.bool(), codes, self.reset_modes))
        o = None
        if one_starting is not None:
            o = self._per_env(one_starting, torch.int8, "one_starting")
        sd = None
        if seed is not None:
            if isinstance(seed, (int, np.integer)) and not isinstance(seed, bool):
                sd = (torch.arange(self.num_envs, dtype=torch.int64, device=self.device) + int(seed)) & 0x7FFFFFFFFFFFFFFF
            else:
                sd = self._per_env(seed, torch.int64, "seed")
        with torch.cuda.device(self.device):
            _lib.check(self.L.hk_reset_seeded(self._h, _ptr(m), _ptr(o), _ptr(sd), None, self._stream()))
            _lib.check(self.L.hk_get_obs(self._h, _ptr(self.obs), _ptr(self.obs2), self._stream()))
            _lib.check(self.L.hk_get_info(self._h, _ptr(self.info), _ptr(self.info2), self._stream()))
            if m is not None or o is not None or sd is not None or mode is not None:
                torch.cuda.current_stream(self.device).synchronize()  # the argument tensors may be temporaries
        return self.obs, self._info_dict(self.info)

    def step(self, action=None):
        """HockeyEnv.step (hockey_env.py:658-695).  action: float32 CUDA tensor [N, 8] (both players), [N, 4]
        (player 1 only, player 2 in-kernel) or None (both in-kernel).  Returns the reference's 5-tuple of
        device tensors: obs [N,18], reward [N], done [N] (uint8), truncated [N] (all False), info dict."""
        a, stride = None, 0
        if self.p1 == _lib.POLICY_EXTERNAL or self.p2 in (_lib.POLICY_EXTERNAL, _lib.POLICY_PER_ENV):
            if action is None:
                raise ValueError("step() needs an action tensor: at least one player is external")
            a = action
            if not (isinstance(a, torch.Tensor) and a.is_cuda and a.dtype == torch.float32 and a.is_contiguous()):
                a = torch.as_tensor(action, dtype=torch.float32, device=self.device).contiguous()
            if a.dim() != 2 or a.shape[0] != self.num_envs:
                raise ValueError(f"action must be [num_envs, 4 or 8], got {tuple(a.shape)}")
            stride = a.shape[1]
            if self.p2 == _lib.POLICY_PER_ENV and stride != 8:
                raise ValueError("p2='per_env' needs [num_envs, 8] actions (columns 4..7 for the external-opponent envs)")
            if self.p2 == _lib.POLICY_EXTERNAL and self.p1 != _lib.POLICY_EXTERNAL and stride == 4:
                # only player 2 is external: its 4 columns are expected at offset 4
                a = torch.cat([torch.zeros_like(a), a], dim=1).contiguous()
                stride = 8
        with torch.cuda.device(self.device):
            _lib.check(self.L.hk_step(self._h, _ptr(a), stride, self.p1, self.p2,
                                      _lib.STEP_AUTORESET if self.auto_reset else 0,
                                      _ptr(self.obs), _ptr(self.obs2), _ptr(self.reward), _ptr(self.reward2),
                                      _ptr(self.done), _ptr(self.info), _ptr(self.info2), _ptr(self.final_obs),
                                      self._stream()))
        return self.obs, self.reward, self.done, self.truncated, self._info_dict(self.info)

    # -- host-agent path: actions from, and results into, pinned host memory ---------------------------------------------
    def host_buffers(self, final_obs=False):
        """One pinned host allocation laid out as obs [N,18] f32 | reward [N] f32 | info [N,4] f32 | done [N] u8
        (| final_obs [N,18] f32) (hk_host_record_bytes), a device record of the same layout and a device action buffer:
        what `step_host` fills.  Returns a dict; rec["host"] / rec["dev"] hold the tensor views."""
        n = self.num_envs
        off = (C.c_int64 * 5)()
        total = int(self.L.hk_host_record_bytes(n, int(bool(final_obs)), off))
        off = list(off)
        raw = torch.empty(total, dtype=torch.uint8).pin_memory()
        dev = torch.empty(total, dtype=torch.uint8, device=self.device)

        def views(buf):
            v = {"obs": buf[off[0]:off[0] + 72 * n].view(torch.float32).view(n, 18),
                 "reward": buf[off[1]:off[1] + 4 * n].view(torch.float32),
                 "info": buf[off[2]:off[2] + 16 * n].view(torch.float32).view(n, 4),
                 "done": buf[off[3]:off[3] + n]}
            v["final_obs"] = buf[off[4]:off[4] + 72 * n].view(torch.float32).view(n, 18) if final_obs else None
            return v
        return {"raw": raw, "host": views(raw), "dev_raw": dev, "dev": views(dev), "final_obs": bool(final_obs),
                "act": torch.empty((n, 8 if self.action_dim == 8 else 4), dtype=torch.float32, device=self.device)}

    def host_bytes_per_step(self, final_obs=False):
        return self.num_envs * (72 + 4 + 16 + 1 + (72 if final_obs else 0))

    def step_host(self, action_host, rec, sync=True, mode="copy"):
        """One tick for a HOST-side agent (the reference's calling pattern): `action_host` (pinned float32 [N,4|8], or None
        when both players are in-kernel) goes to the device, the tick runs, and obs / reward / info / done (/ final_obs)
        arrive in `rec["host"]` (pinned; see host_buffers).  mode:
          "copy"      (default) plain step into the packed device record, then ONE device-to-host copy;
          "overlap"   (hk_step_host) the fast tier's rows travel by DMA while the general tier runs, the general tier
                      stores its rows straight into the mapped host record once that copy has landed;
          "zero_copy" every kernel stores its outputs straight into the mapped host record.
        Measured on B200 / PCIe 5 at 65,536 envs (profiles/README.md): copy 0.72 ms per tick, overlap 0.75, zero_copy 0.86
        against 0.59 for the device-resident step -- scattered 8-byte stores over PCIe cost more than the 0.11 ms DMA.
        sync=True waits for the results.  Returns the reference's 5-tuple as pinned host tensors."""
        if action_host is not None and not (action_host.dtype == torch.float32 and action_host.is_contiguous()
                                            and tuple(action_host.shape) == tuple(rec["act"].shape)):
            raise ValueError(f"action_host must be a contiguous float32 tensor {tuple(rec['act'].shape)}")
        flags = _lib.STEP_AUTORESET if self.auto_reset else 0
        with torch.cuda.device(self.device):
            if mode == "overlap":
                _lib.check(self.L.hk_step_host(self._h, _ptr(action_host), rec["act"].shape[1], self.p1, self.p2, flags,
                                               _ptr(rec["act"]), _ptr(rec["dev_raw"]), _ptr(rec["raw"]),
                                               int(rec["final_obs"]), self._stream()))
            else:
                if action_host is not None:
                    rec["act"].copy_(action_host, non_blocking=True)
                out = rec["host"] if mode == "zero_copy" else rec["dev"]
                _lib.check(self.L.hk_step(self._h, _ptr(rec["act"]) if action_host is not None else None, rec["act"].shape[1],
                                          self.p1, self.p2, flags, _ptr(out["obs"]), None, _ptr(out["reward"]), None,
                                          _ptr(out["done"]), _ptr(out["info"]), None, _ptr(out["final_obs"]), self._stream()))
                if mode != "zero_copy":
                    rec["raw"].copy_(rec["dev_raw"], non_blocking=True)
        if sync:
            torch.cuda.current_stream(self.device).synchronize()
        h = rec["host"]
        return h["obs"], h["reward"], h["done"], self.truncated, self._info_dict(h["info"])

    def rollout(self, k_steps, p1="strong", p2="strong", write_obs=False):
        """k fused ticks in one launch with in-kernel policies and auto-reset (hk_rollout)."""
        with torch.cuda.device(self.device):
            _lib.check(self.L.hk_rollout(self._h, int(k_steps), _policy_id(p1), _policy_id(p2),
                                         _ptr(self.obs) if write_obs else None, self._stream()))

    def obs_agent_two(self):
        """hockey_env.py:500-516 for the current state."""
        if self.obs2 is None:
            self.obs2 = torch.empty((self.num_envs, 18), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.L.hk_get_obs(self._h, None, _ptr(self.obs2), self._stream()))
        return self.obs2

    def get_info_agent_two(self):
        """hockey_env.py:568-591 (needs want_agent_two=True so that the step kernel materialises it)."""
        if self.info2 is None:
            raise ValueError("construct HockeyVecEnv(want_agent_two=True) to get agent-two info/reward")
        return self._info_dict(self.info2)

    def get_reward(self, info=None):
        return self.reward

    def get_reward_agent_two(self, info_two=None):
        if self.reward2 is None:
            raise ValueError("construct HockeyVecEnv(want_agent_two=True) to get agent-two info/reward")
        return self.reward2

    def set_state(self, state):
        """HockeyEnv.set_state (hockey_env.py:594-608): [N,18] visible values; hidden state untouched."""
        s = torch.as_tensor(state, dtype=torch.float32, device=self.device).contiguous()
        if s.shape != (self.num_envs, 18):
            raise ValueError("state must be [num_envs, 18]")
        with torch.cuda.device(self.device):
            _lib.check(self.L.hk_set_obs_state(self._h, _ptr(s), self._stream()))
            torch.cuda.current_stream(self.device).synchronize()  # `s` may be a temporary

    def get_full_state(self):
        """Superset of set_state: the canonical [N, STATE_WORDS] int32 record incl. hidden state."""
        s = torch.empty((self.num_envs, _lib.STATE_WORDS), dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.L.hk_get_state(self._h, _ptr(s), self._stream()))
        return s

    def set_full_state(self, s):
        s = torch.as_tensor(s, device=self.device).to(torch.int32).contiguous()
        if s.shape != (self.num_envs, _lib.STATE_WORDS):
            raise ValueError(f"state must be [num_envs, {_lib.STATE_WORDS}]")
        with torch.cuda.device(self.device):
            _lib.check(self.L.hk_set_state(self._h, _ptr(s), self._stream()))
            torch.cuda.current_stream(self.device).synchronize()

    def current_obs(self):
        with torch.cuda.device(self.device):
            _lib.check(self.L.hk_get_obs(self._h, _ptr(self.obs), None, self._stream()))
        return self.obs

    def stats(self):
        """Episode statistics accumulated on the device (include/hockey_b200.h hk_get_stats)."""
        out = (C.c_double * _lib.STATS_DIM)()
        with torch.cuda.device(self.device):
            _lib.check(self.L.hk_get_stats(self._h, out, self._stream()))
        v = np.array(out[:], dtype=np.float64)
        keys = ["episodes", "wins", "losses", "draws", "env_steps", "sum_return_p1", "sum_return_p2", "sum_return_sq_p1",
                "sum_episode_len", "touches_p1", "touches_p2", "velocity_iterations", "toi_events", "overflows", "general_tier_env_steps"]
        return dict(zip(keys, v.tolist()))

    def kernel_timing(self, enable=True):
        """Record CUDA events around every kernel of the following ticks (measurement only, see hk_kernel_timing)."""
        with torch.cuda.device(self.device):
            _lib.check(self.L.hk_kernel_timing(self._h, int(bool(enable))))

    def kernel_times(self):
        """({'k_fast': ms, 'k_touch': ms, 'k_general': ms, 'k_general2': ms} summed over the recorded ticks, ticks)."""
        out = (C.c_double * 4)()
        steps = C.c_int64(0)
        with torch.cuda.device(self.device):
            _lib.check(self.L.hk_kernel_times(self._h, out, C.byref(steps)))
        return dict(zip(("k_fast", "k_touch", "k_general", "k_general2"), list(out))), int(steps.value)

    def launches_per_step(self):
        """Kernels one step() launches (k_fast, k_touch and the general tier(s) of the cascade)."""
        return int(self.L.hk_launches_per_step(self._h))

    def stats_tensor(self):
        """The device accumulators as a float64 tensor view-copy (for an NCCL all-reduce)."""
        t = torch.empty(_lib.STATS_DIM, dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.L.hk_copy_stats(self._h, _ptr(t), self._stream()))
        return t

    def clear_stats(self):
        with torch.cuda.device(self.device):
            _lib.check(self.L.hk_clear_stats(self._h, self._stream()))

    @staticmethod
    def discrete_to_continous_action(discrete_action, keep_mode=True):
        """hockey_env.py:637-656."""
        a = [(discrete_action == 1) * -1.0 + (discrete_action == 2) * 1.0,
             (discrete_action == 3) * -1.0 + (discrete_action == 4) * 1.0,
             (discrete_action == 5) * -1.0 + (discrete_action == 6) * 1.0]
        if keep_mode:
            a.append((discrete_action == 7) * 1.0)
        return a


class _Box:
    """Minimal stand-in for gymnasium.spaces.Box when gymnasium is not installed."""

    def __init__(self, low, high, shape, dtype=np.float32):
        self.low = np.full(shape, low, dtype=dtype)
        self.high = np.full(shape, high, dtype=dtype)
        self.shape = tuple(shape)
        self.dtype = np.dtype(dtype)

    def sample(self):
        lo = np.where(np.isfinite(self.low), self.low, -1.0)
        hi = np.where(np.isfinite(self.high), self.high, 1.0)
        return np.random.uniform(lo, hi).astype(self.dtype)

    def contains(self, x):
        x = np.asarray(x)
        return x.shape == self.shape and bool(np.all(x >= self.low) and np.all(x <= self.high))


class _Discrete:
    def __init__(self, n):
        self.n = n

    def sample(self):
        return int(np.random.randint(self.n))


try:  # use the real spaces when gymnasium exists (the reference subclasses gym.Env, hockey_env.py:83)
    from gymnasium import spaces as _spaces
    import gymnasium as _gym
    _EnvBase = _gym.Env
    _mkbox = lambda lo, hi, shape: _spaces.Box(lo, hi, shape=shape, dtype=np.float32)
    _mkdisc = lambda n: _spaces.Discrete(n)
except Exception:  # pragma: no cover - depends on the environment
    _EnvBase = object
    _mkbox = lambda lo, hi, shape: _Box(lo, hi, shape)
    _mkdisc = lambda n: _Discrete(n)


class HockeyEnv(_EnvBase):
    """Drop-in for hockey.hockey_env.HockeyEnv (hockey_env.py:83-779): one env, numpy in / numpy out,
    same constructor, same return shapes; physics runs in the CUDA library (batch of 1)."""

    metadata = {"render.modes": ["human", "rgb_array"], "render_fps": FPS}
    continuous = False

    def __init__(self, keep_mode: bool = True, mode=Mode.NORMAL, verbose: bool = False, device="cuda:0", seed=None,
                 _p2=None):
        self.mode = mode
        self.keep_mode = keep_mode
        self.verbose = verbose
        self.timeStep = 1.0 / FPS
        self.done = False
        self.winner = 0
        self.closest_to_goal_dist = 1000
        seed = int(np.random.SeedSequence().entropy % (1 << 63)) if seed is None else int(seed)
        self._vec = HockeyVecEnv(1, mode=self._mode, keep_mode=keep_mode, device=device, seed=seed, auto_reset=False,
                                 p2=_p2, want_agent_two=True)
        self._vec_mode = self._mode  # the mode the library resets the env in
        self.max_timesteps = self._vec.max_timesteps
        self.time = 0
        self.one_starts = True
        obs_dim = 18 if keep_mode else 16
        self.observation_space = _mkbox(-np.inf, np.inf, (obs_dim,))
        self.num_actions = 3 if not keep_mode else 4
        self.action_space = _mkbox(-1, +1, (self.num_actions * 2,))
        self.discrete_action_space = _mkdisc(7)
        self._info = None
        self._info2 = None

    # mode property with the reference's accepted forms and errors (hockey_env.py:754-779)
    @property
    def mode(self):
        return self._mode

    @mode.setter
    def mode(self, value):
        """Takes effect at the next reset, as in the reference (reset reads it, hockey_env.py:357-364)."""
        self._mode = _as_mode(value)

    def seed(self, seed=None):
        """hockey_env.py:157-160: the seed of the NEXT reset's draws (None = the env's own running stream)."""
        self._seed = None if seed is None else int(seed) & 0x7FFFFFFFFFFFFFFF
        return [seed]

    def _obs_np(self, t):
        o = t[0].detach().cpu().numpy().astype(np.float64)  # the reference returns float64 (np.hstack)
        return o if self.keep_mode else o[:16]

    def _info_np(self, t):
        v = t[0].detach().cpu().numpy()
        return {"winner": int(v[0]), "reward_closeness_to_puck": float(v[1]), "reward_touch_puck": float(v[2]),
                "reward_puck_direction": float(v[3])}

    def reset(self, one_starting=None, mode=None, seed=None, options=None):
        if mode is not None:
            self.mode = mode
        self.max_timesteps = 250 if self._mode == Mode.NORMAL else 80
        new_mode = None
        if self._mode != self._vec_mode:
            new_mode = self._vec_mode = self._mode
        if self._mode == Mode.NORMAL:
            self.one_starts = bool(one_starting) if one_starting is not None else (not self.one_starts)
        if seed is not None:
            self.seed(seed)
        pending = getattr(self, "_seed", None)
        self._seed = None
        self._vec.reset(one_starting=self.one_starts if self._mode == Mode.NORMAL else None,
                        seed=None if pending is None else torch.tensor([pending], dtype=torch.int64), mode=new_mode)
        self.done = False
        self.winner = 0
        self.time = 0
        self.closest_to_goal_dist = 1000
        obs = self._obs_np(self._vec.obs)
        self._info = self._info_np(self._vec.info)
        self._info2 = self._info_np(self._vec.info2)
        return obs, dict(self._info)

    def _pad_action(self, action):
        a = np.clip(np.asarray(action, dtype=np.float64), -1, +1).astype(np.float32)
        if not self.keep_mode:  # 3 per player -> 4 per player with shoot = 0
            a = np.concatenate([a[0:3], [0.0], a[3:6], [0.0]]).astype(np.float32)
        return a

    def step(self, action):
        a = self._pad_action(action)
        at = torch.from_numpy(a.reshape(1, -1)).to(self._vec.device)
        obs, reward, done, _, _ = self._vec.step(at)
        self._info = self._info_np(self._vec.info)
        self._info2 = self._info_np(self._vec.info2)
        self._reward2 = float(self._vec.reward2[0].item())
        self.done = bool(done[0].item())
        self.winner = self._info["winner"]
        self.time += 1
        return self._obs_np(obs), float(reward[0].item()), self.done, False, dict(self._info)

    def obs_agent_two(self):
        return self._obs_np(self._vec.obs_agent_two())

    def get_info_agent_two(self):
        return dict(self._info2)

    def _compute_reward(self):
        r = 0
        if self.done:
            if self.winner == 1:
                r += 10
            elif self.winner == -1:
                r -= 10
        return float(r)

    def get_reward(self, info):
        return float(self._compute_reward() + info["reward_closeness_to_puck"])

    def get_reward_agent_two(self, info_two):
        return float(-self._compute_reward() + info_two["reward_closeness_to_puck"])

    def set_state(self, state):
        s = np.zeros(18, dtype=np.float64)
        st = np.asarray(state, dtype=np.float64)
        s[:len(st)] = st
        self._vec.set_state(torch.from_numpy(s.astype(np.float32).reshape(1, 18)))

    def discrete_to_continous_action(self, discrete_action):
        return HockeyVecEnv.discrete_to_continous_action(discrete_action, self.keep_mode)

    def render(self, mode="human"):
        raise NotImplementedError("rendering (pygame, hockey_env.py:697-744) is out of scope of the B200 hot path")

    def close(self):
        self._vec.close()


class BasicOpponent:
    """hockey_env.py:781-833: the scripted PD opponent.  `act` takes one observation (array-like [18], returns a numpy
    float64 action like the reference and advances `phase` with the global numpy RNG as the reference does) or a batch
    (torch tensor [N,18], returns a float32 tensor [N,4] on the same device; per-env phases, torch RNG).  Both go
    through one vectorised controller; inside `HockeyVecEnv` the same rule runs in the step kernel (p1/p2='weak'|'strong')."""

    # per-axis gains relative to kp and braking horizons of the (x, y, angle) PD loop (hockey_env.py:799-801,826-829)
    _KP_SCALE = (1.0, 1.0 / 5, 1.0 / 2)
    _BRAKE_HORIZON = (0.1, 0.1, 1.0)

    def __init__(self, weak=True, keep_mode=True):
        self.weak = weak
        self.keep_mode = keep_mode
        self.phase = np.random.uniform(0, np.pi)

    def _controller(self, o, phase):
        """o: float64 [N,18], phase: float64 [N] (already advanced) -> float64 [N,3 or 4]."""
        kp, kd = (0.5 if self.weak else 10.0), 0.5
        me, vel = o[:, 0:3], o[:, 3:6]
        puck_x, puck_y, puck_vx, puck_vy = o[:, 12], o[:, 13], o[:, 14], o[:, 15]
        home_x = torch.full_like(puck_x, -210 / SCALE)
        incoming = puck_vx < 30.0 / SCALE                      # puck not moving away fast: track it, else go home
        in_reach = (me[:, 0] < puck_x) & ((me[:, 1] - puck_y).abs() < 30.0 / SCALE)
        gap = torch.sqrt((me[:, 0] - puck_x) ** 2 + (me[:, 1] - puck_y) ** 2)
        goal_x = torch.where(incoming & in_reach, puck_x + 0.2, home_x)
        goal_y = torch.where(incoming, torch.where(in_reach, puck_y + puck_vy * gap * 0.1, puck_y), torch.zeros_like(puck_y))
        goal = torch.stack([goal_x, goal_y, MAX_ANGLE * torch.sin(phase)], 1)
        err = goal - me
        gains = torch.tensor(self._KP_SCALE, dtype=o.dtype, device=o.device) * kp
        horizon = torch.tensor(self._BRAKE_HORIZON, dtype=o.dtype, device=o.device)
        brake = ((err / (vel + 0.01)).abs() < horizon).to(o.dtype)
        out = torch.clamp(err * gains - vel * brake * kd, -1, 1)
        if self.keep_mode:
            shoot = ((o[:, 16] > 0) & (o[:, 16] < 7)).to(o.dtype)
            out = torch.cat([out, shoot[:, None]], 1)
        return out

    def act(self, obs, verbose=False):
        if isinstance(obs, torch.Tensor) and obs.dim() == 2:
            return self._act_batch(obs)
        o = torch.as_tensor(np.asarray(obs, dtype=np.float64)).reshape(1, -1)
        self.phase += np.random.uniform(0, 0.2)
        return self._controller(o, torch.tensor([float(self.phase)], dtype=torch.float64))[0].numpy()

    def _act_batch(self, obs):
        n = obs.shape[0]
        if not isinstance(self.phase, torch.Tensor) or self.phase.shape[0] != n:
            self.phase = torch.rand(n, dtype=torch.float64, device=obs.device) * math.pi
        self.phase = self.phase + torch.rand(n, dtype=torch.float64, device=obs.device) * 0.2
        return self._controller(obs.to(torch.float64), self.phase).to(torch.float32)


class HockeyEnv_BasicOpponent(HockeyEnv):
    """hockey_env.py:875-886: player 2 is a BasicOpponent; here it runs inside the step kernel."""

    def __init__(self, mode=Mode.NORMAL, weak_opponent=False, device="cuda:0", seed=None):
        super().__init__(mode=mode, keep_mode=True, device=device, seed=seed, _p2="weak" if weak_opponent else "strong")
        self.opponent = BasicOpponent(weak=weak_opponent)  # API compatibility; acting happens in-kernel
        self.action_space = _mkbox(-1, +1, (4,))

    def step(self, action):
        a = np.clip(np.asarray(action, dtype=np.float64), -1, +1).astype(np.float32)
        at = torch.from_numpy(a.reshape(1, 4)).to(self._vec.device)
        obs, reward, done, _, _ = self._vec.step(at)
        self._info = self._info_np(self._vec.info)
        self._info2 = self._info_np(self._vec.info2)
        self.done = bool(done[0].item())
        self.winner = self._info["winner"]
        self.time += 1
        return self._obs_np(obs), float(reward[0].item()), self.done, False, dict(self._info)


class PolicyOpponent:
    """hockey_env.py:908-922: adapts a torch policy to the opponent protocol `act(obs) -> action`.  One observation
    (array-like [18]) gives a numpy action like the reference; a batch tensor [N,18] gives a tensor on its device."""

    def __init__(self, policy, device=None):
        self.policy = policy
        self.device = device

    @torch.no_grad()
    def act(self, obs):
        if isinstance(obs, torch.Tensor) and obs.dim() == 2:
            return self.policy(obs.to(dtype=torch.float32, device=self.device or obs.device))
        row = torch.as_tensor(np.asarray(obs), dtype=torch.float32, device=self.device)[None]
        return self.policy(row)[0].cpu().numpy()


# ---- env registry (hockey_env.py:889-903) ------------------------------------------------------------------------
# The reference registers 'Hockey-v0' and 'Hockey-One-v0' with gymnasium; the same ids resolve here through make()
# (and through gymnasium.make as well when gymnasium is installed), with the reference's default kwargs.
REGISTRY = {
    "Hockey-v0": ("HockeyEnv", {"mode": 0}),
    "Hockey-One-v0": ("HockeyEnv_BasicOpponent", {"mode": 0, "weak_opponent": False}),
}


def spec(env_id):
    """(class, default kwargs) registered under `env_id`."""
    try:
        name, kwargs = REGISTRY[env_id]
    except KeyError:
        raise ValueError(f"unknown env id {env_id!r}; registered: {sorted(REGISTRY)}")
    return globals()[name], dict(kwargs)


def make(env_id, **kwargs):
    """gymnasium.make for the two registered ids: make('Hockey-One-v0', mode=Mode.TRAIN_DEFENSE, weak_opponent=True)."""
    cls, defaults = spec(env_id)
    defaults.update(kwargs)
    return cls(**defaults)


def make_vec(env_id, num_envs, **kwargs):
    """Batched form of make(): the HockeyGymVectorEnv a SyncVectorEnv of `num_envs` such envs would be."""
    from .vector import HockeyGymVectorEnv
    cls, defaults = spec(env_id)
    defaults.update(kwargs)
    opponent = None
    if cls is HockeyEnv_BasicOpponent:
        opponent = "weak" if defaults.pop("weak_opponent", False) else "strong"
    return HockeyGymVectorEnv(num_envs, mode=defaults.pop("mode", Mode.NORMAL), opponent=opponent, **defaults)


try:  # optional: only when gymnasium is importable (it is not part of this image)
    from gymnasium.envs.registration import register as _gym_register
    for _id, (_name, _kw) in REGISTRY.items():
        try:
            _gym_register(id=_id, entry_point=f"hockey_env_b200.env:{_name}", kwargs=dict(_kw))
        except Exception as _e:  # already registered (e.g. by the reference package)
            pass
except ImportError:
    pass
