"""gymnasium.vector.VectorEnv over HockeyVecEnv (SURVEY.md section 8f, rank 1).

What `gymnasium.vector.SyncVectorEnv([lambda: HockeyEnv_BasicOpponent(...)] * n, autoreset_mode=SAME_STEP)` gives a
caller of the reference (hockey_env.py:875-903), as one batched env on the GPU:

  * `num_envs`, `single_observation_space`, `single_action_space`, batched `observation_space` / `action_space`;
  * `reset(seed=, options=) -> (obs, infos)`: seed = None / int (env i gets seed + i, gymnasium's convention) / list of
    ints; options may hold "reset_mask" (bool [N], gymnasium >= 1.1), "one_starting" and "mode" (the reference's reset
    arguments; "mode" is one Mode or one per env and also governs the later auto-resets of the reset envs);
  * `step(actions) -> (obs, rewards, terminations, truncations, infos)` with SAME-STEP auto-reset: the returned obs of a
    finished env is the first obs of its next episode, its terminal observation is infos["final_obs"][i] and its
    terminal info (winner, reward terms) infos["final_info"][key][i], selected by the boolean masks infos["_final_obs"]
    / infos["_final_info"]; `truncations` is always False (the reference never truncates, hockey_env.py:695).

It IS a `gymnasium.vector.VectorEnv` when gymnasium is importable, and works unchanged without it.
"""
import numpy as np
import torch

from .env import HockeyVecEnv, Mode, _mkbox

try:  # pragma: no cover - depends on the environment (gymnasium is not part of this image)
    from gymnasium.vector import VectorEnv as _VectorEnvBase
    try:
        from gymnasium.vector import AutoresetMode as _AutoresetMode
        _SAME_STEP = _AutoresetMode.SAME_STEP
    except Exception:
        _SAME_STEP = "same_step"
except Exception:
    _VectorEnvBase = object
    _SAME_STEP = "same_step"

_INFO_KEYS = ("winner", "reward_closeness_to_puck", "reward_touch_puck", "reward_puck_direction")


class HockeyGymVectorEnv(_VectorEnvBase):
    metadata = {"autoreset_mode": _SAME_STEP, "render_modes": []}
    render_mode = None
    spec = None

    def __init__(self, num_envs, mode=Mode.NORMAL, opponent="strong", device="cuda:0", seed=0, numpy_io=True, keep_mode=True):
        """opponent: 'weak' / 'strong' (HockeyEnv_BasicOpponent semantic, 4-d actions) or None (HockeyEnv, 8-d actions).
        mode: one Mode for all envs or one per env (HockeyVecEnv)."""
        self.env = HockeyVecEnv(num_envs, mode=mode, keep_mode=keep_mode, device=device, seed=seed, auto_reset=True, p2=opponent)
        self.num_envs = int(num_envs)
        self.numpy_io = bool(numpy_io)
        act = 4 if opponent else 8
        self.single_observation_space = _mkbox(-np.inf, np.inf, (18,))
        self.single_action_space = _mkbox(-1, +1, (act,))
        self.observation_space = _mkbox(-np.inf, np.inf, (self.num_envs, 18))
        self.action_space = _mkbox(-1, +1, (self.num_envs, act))
        self.closed = False

    @property
    def unwrapped(self):
        return self

    def _out(self, t):
        return t.detach().cpu().numpy() if self.numpy_io else t

    def _infos(self, done=None):
        e = self.env
        infos = {k: self._out(e.info[:, c]) for c, k in enumerate(_INFO_KEYS)}
        if done is not None:
            mask = self._out(done.to(torch.bool))
            infos["final_obs"] = self._out(e.final_obs)
            infos["_final_obs"] = mask
            # the info tensor of a tick is written before the auto-reset: on a finished env it IS the terminal info
            infos["final_info"] = {k: infos[k] for k in _INFO_KEYS}
            infos["_final_info"] = mask
        return infos

    def reset(self, *, seed=None, options=None):
        options = options or {}
        if seed is not None and not isinstance(seed, (int, np.integer)):
            seed = np.asarray([-1 if s is None else int(s) for s in seed], dtype=np.int64)
        obs, _ = self.env.reset(mask=options.get("reset_mask"), one_starting=options.get("one_starting"), seed=seed,
                                mode=options.get("mode"))
        return self._out(obs), self._infos()

    def step(self, actions):
        a = torch.as_tensor(actions, dtype=torch.float32, device=self.env.device)
        obs, reward, done, trunc, _ = self.env.step(a.contiguous())
        return (self._out(obs), self._out(reward), self._out(done.to(torch.bool)), self._out(trunc), self._infos(done))

    def close(self, **kwargs):
        if not self.closed:
            self.env.close()
            self.closed = True

    def close_extras(self, **kwargs):
        self.close()
