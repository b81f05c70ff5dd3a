"""Device-side plumbing around the hot path for the reference's training loop -- SURVEY.md section 8f, ranks 2-4.

Everything here consumes and produces the env's zero-copy device tensors; nothing makes a host round trip per tick.
The dense networks are plain torch modules (library matmuls): they are the ops next to the hot path, not the path.

* `OpponentPool`        per-env opponent selection: weak / strong BasicOpponent (in-kernel) or self-play snapshots
                        (batched actor inference on obs_agent_two()), re-drawn per episode
                        (rl/training/opponent_manager.py:19-91, rl/training/self_play.py:7-68, hockey_env.py:908-922)
* `ModeMix`             per-env game mode: NORMAL / TRAIN_SHOOTING / TRAIN_DEFENSE drawn per episode from probabilities
                        that may change between calls (curriculum), with per-mode win / loss / draw counters on the device
* `DeviceReplayBuffer`  ring buffer in HBM fed straight from step outputs (rl/replay/base_buffer.py:21-41,
                        rl/replay/uniform_buffer.py) -- `push` is one batched copy per tick instead of N Python calls
* `evaluate`            the Evaluator protocol (rl/utils/evaluator.py:10-35): win / draw / loss rates and mean return
                        of a policy against a fixed opponent over n COMPLETE episodes (fixed quota per env)
* `cross_play`          league table: K actors against each other (K x K ordered pairs) in one batch, one pooled
                        tensor-core launch per player per tick, with `evaluate`'s complete-episode protocol
* `evaluate_model`      the ModelEvaluator protocol (model_evaluation/model_evaluator.py:81-108): 300 episodes, seed
                        123, against the weak and the strong BasicOpponent
"""
import torch

from . import _lib
from .actor import ExplorationNoise, FusedActor, FusedActorPool
from .env import HockeyVecEnv, Mode


class OpponentPool:
    """Draws, per env and per episode, one opponent out of {weak, strong, snapshot_0..k-1} with the given
    probabilities (the reference draws one per episode for its single env; here every env of the batch holds its own
    draw).  BasicOpponents run inside the step kernel.  Snapshot opponents are either a list of modules (each evaluated
    on `obs_agent_two()` for all envs at once; their actions are only read by the envs that drew them) or a
    `FusedActorPool`: then one pooled tensor-core launch evaluates, per env, only the snapshot it drew, straight into
    columns 4..7 of a persistent [N, 8] action buffer."""

    WEAK, STRONG, SNAPSHOT0 = 0, 1, 2

    def __init__(self, env, p_weak=0.5, p_strong=0.5, snapshots=(), p_snapshot=0.0, seed=0):
        if env.p2 != _lib.POLICY_PER_ENV:
            raise ValueError("OpponentPool needs HockeyVecEnv(..., p2='per_env')")
        self.env = env
        self.fused = isinstance(snapshots, FusedActorPool)
        self.snapshots = snapshots if self.fused else list(snapshots)
        if p_snapshot > 0 and not self.snapshots:
            raise ValueError("p_snapshot > 0 without snapshots")
        k = len(self.snapshots)
        probs = [p_weak, p_strong] + [p_snapshot / k] * k
        self.probs = torch.tensor(probs, dtype=torch.float32, device=env.device)
        self.probs = self.probs / self.probs.sum()
        self.gen = torch.Generator(device=env.device)
        self.gen.manual_seed(seed)
        self.choice = torch.zeros(env.num_envs, dtype=torch.long, device=env.device)
        self.codes = env.opponent_codes
        self._a2 = torch.zeros((env.num_envs, 4), dtype=torch.float32, device=env.device)
        if self.fused:
            self._a8 = torch.zeros((env.num_envs, 8), dtype=torch.float32, device=env.device)
            self._pick = torch.empty(env.num_envs, dtype=torch.int32, device=env.device)
        self.resample(None)

    def add_snapshot(self, actor, p_snapshot=None):
        """SelfPlayManager.add_snapshot (rl/training/self_play.py:30-45): later draws may pick `actor` (a module; with a
        `FusedActorPool` it is packed into the pool)."""
        if self.fused:
            self.snapshots.add(actor)
        else:
            self.snapshots.append(actor)
        k = len(self.snapshots)
        ps = float(self.probs[2:].sum()) if p_snapshot is None else float(p_snapshot)
        base = self.probs[:2] / self.probs[:2].sum() * (1.0 - ps)
        self.probs = torch.cat([base, torch.full((k,), ps / k, device=self.env.device)])

    def resample(self, done):
        """Re-draw the opponent of every env whose episode just ended (`done` = the step's done tensor, None = all)."""
        n = self.env.num_envs
        draw = torch.multinomial(self.probs.expand(n, -1), 1, generator=self.gen).squeeze(1)
        if done is None:
            self.choice.copy_(draw)
        else:
            self.choice.copy_(torch.where(done.to(torch.bool), draw, self.choice))
        code = torch.where(self.choice == self.WEAK, _lib.POLICY_BASIC_WEAK,
                           torch.where(self.choice == self.STRONG, _lib.POLICY_BASIC_STRONG, _lib.POLICY_EXTERNAL))
        self.codes.copy_(code.to(torch.uint8))  # in place: the step kernel reads this very tensor

    @torch.no_grad()
    def opponent_actions(self):
        """[N,4] actions of the snapshot opponents (zeros where an in-kernel BasicOpponent plays)."""
        if not len(self.snapshots):
            return self._a2
        if self.fused:
            a2 = self._a8[:, 4:]
            a2.zero_()
            # snapshot index for the envs that drew one, -1 (not written) for the BasicOpponent envs
            torch.sub(self.choice, self.SNAPSHOT0, out=self._pick).masked_fill_(self.choice < self.SNAPSHOT0, -1)
            return self.snapshots(self.env.obs_agent_two(), self._pick, out=a2)
        obs2 = self.env.obs_agent_two()
        self._a2.zero_()
        for k, actor in enumerate(self.snapshots):
            m = self.choice == self.SNAPSHOT0 + k
            # evaluated for the whole batch (dense, no gather/scatter); only the rows that drew this snapshot are kept
            self._a2 = torch.where(m.unsqueeze(1), actor(obs2), self._a2)
        return self._a2

    def step(self, a1):
        """One env tick with player-1 actions `a1` [N,4]; returns the env's step tuple.  Opponents of finished
        episodes are re-drawn afterwards."""
        if self.fused:
            self.opponent_actions()
            self._a8[:, :4].copy_(a1)
            out = self.env.step(self._a8)
        else:
            out = self.env.step(torch.cat([a1, self.opponent_actions()], dim=1).contiguous())
        self.resample(out[2])
        return out


class ModeMix:
    """Draws, per env and per episode, the game mode out of {NORMAL, TRAIN_SHOOTING, TRAIN_DEFENSE} with probabilities
    `probs` (change them between calls with `set_probs`, e.g. to anneal a curriculum).  The draws go to the env's reset
    codes (`HockeyVecEnv.set_reset_modes`), which the library reads AT each reset: each episode's mode is therefore
    drawn one episode ahead -- when the previous episode of that env starts (or at construction) -- and an auto-reset
    starts the episode in the mode drawn before it.  Call `update(done, winner)` after every step of the env (or use
    `step`); it credits each finished episode to the mode it was played in and re-draws the codes of the envs that
    just auto-reset.  Counters `counts` [3 modes, 4]: episodes, wins, losses, draws (float64, on the device: no host
    sync per tick).  Explicit `env.reset` calls outside `reset` are not seen by the helper."""

    EPISODES, WINS, LOSSES, DRAWS = 0, 1, 2, 3

    def __init__(self, env, probs=(1 / 3, 1 / 3, 1 / 3), seed=0):
        if not env.auto_reset:
            raise ValueError("ModeMix needs HockeyVecEnv(..., auto_reset=True)")
        self.env = env
        self.gen = torch.Generator(device=env.device)
        self.gen.manual_seed(seed)
        self.set_probs(probs)
        self.counts = torch.zeros((3, 4), dtype=torch.float64, device=env.device)
        self.playing = env.modes().clone()  # mode of each env's running episode
        self.codes = env.set_reset_modes(self._draw())  # mode of each env's next episode

    def set_probs(self, probs):
        """Probabilities of NORMAL, TRAIN_SHOOTING, TRAIN_DEFENSE for the draws from now on (normalised)."""
        p = torch.as_tensor(probs, dtype=torch.float32).to(self.env.device).reshape(3)
        if bool((p < 0).any()) or float(p.sum()) <= 0:
            raise ValueError("probs must be three non-negative numbers with a positive sum")
        self.probs = p / p.sum()

    def _draw(self):
        n = self.env.num_envs
        return torch.multinomial(self.probs.expand(n, -1), 1, replacement=True, generator=self.gen).squeeze(1).to(torch.uint8)

    def reset(self, **kwargs):
        """env.reset(**kwargs) of every env (no mask): the episodes it starts play the drawn codes; draws the next ones."""
        if "mask" in kwargs or "mode" in kwargs:
            raise ValueError("ModeMix.reset resets every env in its drawn mode")
        out = self.env.reset(**kwargs)
        self.playing.copy_(self.codes)
        self.codes.copy_(self._draw())
        return out

    def update(self, done, winner):
        """After a step: credit the finished episodes (`done` [N], `winner` = info[:, 0]) to the mode they were played
        in, then let the envs that auto-reset play their code and draw the code of their following episode."""
        d = done.to(torch.bool)
        w = winner.to(torch.float64)
        rows = torch.stack([torch.ones_like(w), (w == 1).to(torch.float64), (w == -1).to(torch.float64),
                            (w == 0).to(torch.float64)], 1) * d.unsqueeze(1).to(torch.float64)
        self.counts.index_add_(0, self.playing.long(), rows)
        self.playing.copy_(torch.where(d, self.codes, self.playing))
        self.codes.copy_(torch.where(d, self._draw(), self.codes))  # in place: the library reads this very tensor

    def step(self, action=None):
        """One env tick followed by `update`; returns the env's step tuple."""
        out = self.env.step(action)
        self.update(out[2], out[4]["winner"])
        return out

    def stats(self):
        """{mode name: {episodes, wins, losses, draws}} (synchronises the host)."""
        c = self.counts.cpu().tolist()
        return {m.name: dict(zip(("episodes", "wins", "losses", "draws"), c[m.value])) for m in Mode}


class DeviceReplayBuffer:
    """Uniform replay buffer in device memory (rl/replay/base_buffer.py, uniform_buffer.py): `push` appends a whole
    batch of transitions (one per env) with five strided copies, `sample` gathers a minibatch with one index tensor."""

    def __init__(self, capacity, obs_dim=18, action_dim=4, device="cuda:0", seed=0):
        self.capacity, self.device = int(capacity), torch.device(device)
        self.obs = torch.empty((self.capacity, obs_dim), dtype=torch.float32, device=self.device)
        self.action = torch.empty((self.capacity, action_dim), dtype=torch.float32, device=self.device)
        self.reward = torch.empty(self.capacity, dtype=torch.float32, device=self.device)
        self.next_obs = torch.empty((self.capacity, obs_dim), dtype=torch.float32, device=self.device)
        self.done = torch.empty(self.capacity, dtype=torch.float32, device=self.device)
        self.pos, self.size = 0, 0
        self.gen = torch.Generator(device=self.device)
        self.gen.manual_seed(seed)

    def __len__(self):
        return self.size

    def push(self, obs, action, reward, next_obs, done):
        """Batch of n transitions (n <= capacity); wraps around like the reference's ring buffer."""
        n = obs.shape[0]
        if n > self.capacity:
            raise ValueError("batch larger than the buffer")
        first = min(n, self.capacity - self.pos)
        for dst, src in ((self.obs, obs), (self.action, action), (self.reward, reward), (self.next_obs, next_obs),
                         (self.done, done.to(torch.float32))):
            dst[self.pos:self.pos + first].copy_(src[:first])
            if first < n:
                dst[:n - first].copy_(src[first:])
        self.pos = (self.pos + n) % self.capacity
        self.size = min(self.capacity, self.size + n)

    def sample_indices(self, batch_size):
        """The int64 row indices `sample` gathers (drawn from the buffer's generator): uniform over the stored rows."""
        return torch.randint(0, self.size, (batch_size,), device=self.device, generator=self.gen)

    def sample(self, batch_size):
        idx = self.sample_indices(batch_size)
        return self.obs[idx], self.action[idx], self.reward[idx], self.next_obs[idx], self.done[idx]


def behaviour_actions(actor, obs, noise=0.0, reset=None):
    """The behaviour policy of one tick: actor(obs), plus Gaussian exploration noise of std `noise` clamped to [-1, 1]
    when noise > 0.  A `FusedActor` draws the noise in its kernel epilogue (one launch); any other module runs, then
    torch's randn / add / clamp.  noise=ExplorationNoise (a `FusedActor` only: its state lives in the fused launch)
    explores through slot 0, with `reset` = the previous step's done tensor (None on the first tick)."""
    if isinstance(noise, ExplorationNoise):
        if not isinstance(actor, FusedActor):
            raise ValueError("noise=ExplorationNoise needs a FusedActor: the noise state exists only in the fused launch")
        return actor(obs, noise=noise, reset=reset)
    if not noise:
        return actor(obs)
    if isinstance(actor, FusedActor):
        return actor(obs, noise=noise)
    a = actor(obs)
    return (a + torch.randn(a.shape, device=a.device) * noise).clamp(-1, 1)


@torch.no_grad()
def collect(pool_or_env, actor, buffer, steps, noise=0.0):
    """`steps` ticks of experience collection: actor -> env -> buffer, all on the device.  `actor` is a module or a
    `FusedActor`; `noise` > 0 adds Gaussian exploration noise of that std (see `behaviour_actions`), an
    `ExplorationNoise` its per-env process, reset for the envs whose episode ended on the previous tick.  With auto-reset
    the transition of a finished episode stores the TERMINAL observation (`final_obs`) as next_obs, as the reference's
    loop does (rl/training/train.py:136-160)."""
    env = pool_or_env.env if isinstance(pool_or_env, OpponentPool) else pool_or_env
    obs = env.obs.clone()
    done = None
    for _ in range(steps):
        a1 = behaviour_actions(actor, obs, noise, reset=done if isinstance(noise, ExplorationNoise) else None)
        nobs, reward, done, _, _ = pool_or_env.step(a1) if isinstance(pool_or_env, OpponentPool) else env.step(a1.contiguous())
        nxt = torch.where(done.to(torch.bool).unsqueeze(1), env.final_obs, nobs) if env.final_obs is not None else nobs
        buffer.push(obs, a1, reward, nxt, done)
        obs = nobs.clone()
    if isinstance(noise, ExplorationNoise) and done is not None:
        noise.reset(done)  # episodes that ended on the last tick start the next call from x = 0
    return buffer


def _play_quota(env, act, k, max_ticks, credit):
    """The complete-episode protocol of `evaluate`: sides alternate per env (even envs start with player 1), every env
    plays a quota of `k` complete episodes and only those count.  Each tick: `act(obs)` gives the step's action tensor;
    `credit(fin, winner, ret, length)` receives the float64 mask of the episodes that just finished within quota, the
    winners, and the returns and lengths of those episodes.  Returns the per-env episode counts and the ticks played."""
    n, dev = env.num_envs, env.device
    obs, _ = env.reset(one_starting=(torch.arange(n, device=dev) % 2 == 0).to(torch.int8))
    count = torch.zeros(n, dtype=torch.int64, device=dev)
    ret = torch.zeros(n, dtype=torch.float64, device=dev)
    length = torch.zeros(n, dtype=torch.int64, device=dev)
    ticks = 0
    while ticks < max_ticks:
        obs, reward, done, _, info = env.step(act(obs))
        ticks += 1
        ret += reward.to(torch.float64)
        length += 1
        fin = done.to(torch.bool) & (count < k)
        credit(fin.to(torch.float64), info["winner"], ret, length)
        count += fin
        ret = torch.where(done.to(torch.bool), torch.zeros_like(ret), ret)
        length = torch.where(done.to(torch.bool), torch.zeros_like(length), length)
        if ticks % 16 == 0 and bool((count >= k).all().item()):  # one small host read every 16 ticks
            break
    return count, ticks


@torch.no_grad()
def evaluate(actor, n_episodes=1000, opponent="strong", mode=Mode.NORMAL, num_envs=4096, device="cuda:0", seed=0,
             max_ticks=100000):
    """Evaluator.evaluate (rl/utils/evaluator.py:10-35) batched: `actor` (obs [N,18] -> actions [N,4]) plays COMPLETE
    episodes of Hockey-One-v0 against the in-kernel weak/strong BasicOpponent; returns the win rate (`winner == 1`) and
    the mean return (sum of step rewards) the reference reports, plus draw/loss rates and the mean episode length.

    Every env plays the same quota of k = ceil(n_episodes / num_envs) complete episodes and only those are counted (an
    env that has filled its quota keeps stepping but is ignored), so k * num_envs >= n_episodes episodes are played --
    stopping all envs once a global count is reached would keep only the shortest episodes and lose the 251-tick
    draws.  Sides alternate like the reference's reset (hockey_env.py:359-362): even envs start with player 1."""
    env = HockeyVecEnv(num_envs, mode=mode, device=device, seed=seed, p2=opponent)
    n = env.num_envs
    k = -(-int(n_episodes) // n)
    acc = torch.zeros(6, dtype=torch.float64, device=env.device)  # wins, draws, losses, sum return, sum return^2, sum length

    def credit(f64, w, ret, length):
        acc.add_(torch.stack([(f64 * (w == 1)).sum(), (f64 * (w == 0)).sum(), (f64 * (w == -1)).sum(), (f64 * ret).sum(),
                              (f64 * ret * ret).sum(), (f64 * length).sum()]))

    count, ticks = _play_quota(env, lambda obs: actor(obs).contiguous(), k, max_ticks, credit)
    env.close()
    a = acc.cpu().tolist()
    m = max(int(count.sum().item()), 1)
    mean_ret = a[3] / m
    return {"episodes": m, "win_rate": a[0] / m, "draw_rate": a[1] / m, "loss_rate": a[2] / m, "mean_return": mean_ret,
            "std_return": max(a[4] / m - mean_ret * mean_ret, 0.0) ** 0.5, "mean_length": a[5] / m, "ticks": ticks,
            "episodes_per_env": k}


@torch.no_grad()
def cross_play(actors, episodes_per_pair, num_envs, mode=Mode.NORMAL, seed=0, device="cuda:0", max_ticks=100000):
    """League table of K actors (modules of the reference architecture, or a `FusedActorPool`): every ordered pair
    (i as player 1, j as player 2) plays `episodes_per_pair` or more COMPLETE episodes on an equal block of
    B = num_envs // K^2 envs (rounded down to even, so both sides start equally often), with `evaluate`'s protocol:
    a quota of ceil(episodes_per_pair / B) episodes per env, alternating sides.  Each tick is two pooled tensor-core
    launches: player 1 on `obs` into action columns 0..3, player 2 on `obs_agent_two()` into columns 4..7.

    Returns [K, K] float64 tensors (row i = player 1, column j = player 2, player 1's side): `win_rate`, `draw_rate`,
    `loss_rate`, `mean_return`, and `episodes`; plus `ticks` and `episodes_per_env`."""
    pool = actors if isinstance(actors, FusedActorPool) else FusedActorPool(actors, device=device)
    kk = len(pool)
    if kk < 1:
        raise ValueError("cross_play needs at least one actor")
    per_pair = num_envs // (kk * kk)
    per_pair -= per_pair % 2
    if per_pair < 2:
        raise ValueError(f"cross_play needs num_envs >= 2 * K^2 = {2 * kk * kk}")
    env = HockeyVecEnv(per_pair * kk * kk, mode=mode, device=pool.device, seed=seed, p1=None, p2=None)
    n, dev = env.num_envs, env.device
    pair = torch.arange(n, device=dev) // per_pair
    c1, c2 = (pair // kk).to(torch.int32), (pair % kk).to(torch.int32)
    a8 = torch.zeros((n, 8), dtype=torch.float32, device=dev)
    acc = torch.zeros((kk * kk, 6), dtype=torch.float64, device=dev)  # per pair: as `evaluate`'s accumulator

    def act(obs):
        pool(obs, c1, out=a8[:, :4])
        pool(env.obs_agent_two(), c2, out=a8[:, 4:])
        return a8

    def credit(f64, w, ret, length):
        acc.index_add_(0, pair, torch.stack([f64 * (w == 1), f64 * (w == 0), f64 * (w == -1), f64 * ret, f64 * ret * ret,
                                             f64 * length], 1))

    k = -(-int(episodes_per_pair) // per_pair)
    count, ticks = _play_quota(env, act, k, max_ticks, credit)
    env.close()
    episodes = torch.zeros(kk * kk, dtype=torch.float64, device=dev).index_add_(0, pair, count.to(torch.float64))
    m = episodes.clamp(min=1).unsqueeze(1)
    rates = (acc / m).view(kk, kk, 6)
    return {"win_rate": rates[..., 0], "draw_rate": rates[..., 1], "loss_rate": rates[..., 2], "mean_return": rates[..., 3],
            "episodes": episodes.view(kk, kk), "ticks": ticks, "episodes_per_env": k}


@torch.no_grad()
def evaluate_model(actor, episodes=300, seed=123, num_envs=None, device="cuda:0"):
    """ModelEvaluator._eval_once for both opponents (model_evaluation/model_evaluator.py:81-108, defaults :234-235:
    300 complete episodes, seed 123): win rate and mean return of `actor` on Hockey-One-v0 against the weak and the
    strong BasicOpponent -- the four numbers of one row of the reference's final-evaluation table."""
    n = int(num_envs) if num_envs else int(episodes)
    weak = evaluate(actor, n_episodes=episodes, opponent="weak", num_envs=n, device=device, seed=seed)
    strong = evaluate(actor, n_episodes=episodes, opponent="strong", num_envs=n, device=device, seed=seed)
    return {"wr_weak": weak["win_rate"], "wr_strong": strong["win_rate"], "ret_weak": weak["mean_return"],
            "ret_strong": strong["mean_return"], "episodes": weak["episodes"]}
