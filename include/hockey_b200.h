/* hockey_b200.h -- C ABI of the B200-native batched HockeyEnv hot path.
 *
 * This is the drop-in boundary for the reference's `HockeyEnv.step()/reset()` path
 * (reference: hockey/hockey_env.py:345-418 reset, :658-695 step, :781-833 BasicOpponent,
 * :594-608 set_state).  The reference crosses Python -> SWIG -> Box2D C++ once per Box2D call
 * (hockey_env.py:682 `self.world.Step(...)` plus ~40 property reads/writes per tick); this library
 * replaces that whole per-tick path with one CUDA launch over a batch of independent envs.
 *
 * Conventions
 *  - plain pointers and sizes only; every `*_dev` pointer is a CUDA device pointer owned by the
 *    CALLER (e.g. a torch tensor's data_ptr()); the library owns only its internal state buffers.
 *  - every entry point returns 0 on success or a negative HK_E_* code; hk_last_error() gives the
 *    message (thread-local).  Nothing throws or exits across the ABI.
 *  - all work is enqueued on the caller's stream (`stream` is a cudaStream_t passed as void*;
 *    NULL = legacy default stream).  No allocation, host sync or host copy happens in
 *    hk_step / hk_reset / hk_rollout, so they are CUDA-graph capturable.
 *  - a handle is not thread-safe; one handle per process/GPU.
 */
#ifndef HOCKEY_B200_H
#define HOCKEY_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct hk_env hk_env;

/* ---- error codes ---------------------------------------------------------------------------- */
enum {
  HK_OK = 0,
  HK_E_INVALID = -1, /* bad argument (mirrors the reference's ValueError/TypeError, hockey_env.py:769-779) */
  HK_E_CUDA = -2,    /* a CUDA runtime call failed */
  HK_E_NODEVICE = -3 /* no CUDA device: there is no CPU fallback */
};

/* ---- modes (reference `class Mode(Enum)`, hockey_env.py:78-81) ------------------------------- */
enum { HK_MODE_NORMAL = 0, HK_MODE_TRAIN_SHOOTING = 1, HK_MODE_TRAIN_DEFENSE = 2 };

/* ---- per-player action source for a tick ---------------------------------------------------- */
enum {
  HK_POLICY_EXTERNAL = 0,     /* read 4 floats from the caller's action tensor                       */
  HK_POLICY_BASIC_WEAK = 1,   /* in-kernel BasicOpponent(weak=True)  (hockey_env.py:781-833)         */
  HK_POLICY_BASIC_STRONG = 2, /* in-kernel BasicOpponent(weak=False)                                 */
  HK_POLICY_RANDOM = 3,       /* U(-1,1)^4 from Philox4x32-10 keyed (seed, global env id, tick)      */
  HK_POLICY_ZERO = 4,         /* all-zero action                                                     */
  HK_POLICY_PER_ENV = 5       /* player 2 only: one of the codes above per env (hk_set_opponent_policies) */
};

/* ---- step flags ----------------------------------------------------------------------------- */
enum {
  HK_STEP_AUTORESET = 1 /* on done: emit terminal reward/done/info, then reset that env in the same
                           launch; `obs` holds the new episode's first observation and `final_obs`
                           (if given) the terminal one.  Off = reference behaviour (stepping after
                           done is allowed, hockey_env.py:658-695 has no guard). */
};

/* ---- sizes ---------------------------------------------------------------------------------- */
#define HK_OBS_DIM 18    /* hockey_env.py:125-144 */
#define HK_ACT_DIM 4     /* per player, keep_mode (hockey_env.py:147-148) */
#define HK_INFO_DIM 4    /* winner, reward_closeness_to_puck, reward_touch_puck, reward_puck_direction
                            (hockey_env.py:562-566), as floats */
#define HK_STATS_DIM 16  /* int64/double accumulators, see hk_get_stats */

/* ---- full-state record (hk_get_state / hk_set_state), 32-bit words per env ------------------ *
 * Everything the next tick depends on, visible (the 18-d obs) and hidden (SURVEY.md A.6).        */
enum {
  HK_S_R1 = 0,        /* 8 f32: origin x,y (b2Body::m_xf.p), centre-of-mass x,y (m_sweep.c), angle, vx, vy, w */
  HK_S_R2 = 8,        /* same for player 2 */
  HK_S_PUCK = 16,     /* 6 f32: cx, cy, angle, vx, vy, w */
  HK_S_SLEEP = 22,    /* 3 f32: b2Body::m_sleepTime of racket1, racket2, puck */
  HK_S_FLAGS = 25,    /* u32: bit0-2 awake (r1,r2,puck); bit3 done; bit4 one_starts; bits5-6 winner+1 */
  HK_S_TIME = 26,     /* i32 self.time */
  HK_S_HAS1 = 27,     /* i32 player1_has_puck */
  HK_S_HAS2 = 28,     /* i32 player2_has_puck */
  HK_S_PFORCE = 29,   /* 2 f32: force pending on the puck (TRAIN_DEFENSE reset shot, hockey_env.py:410-411) */
  HK_S_FAT = 31,      /* 12 f32: broad-phase fat AABBs lo.x,lo.y,hi.x,hi.y of racket1, racket2, puck */
  HK_S_MOVED = 43,    /* u32: buffered broad-phase moves bit0-2 (r1,r2,puck); bit3 = new fixtures (after reset) */
  HK_S_PHASE = 44,    /* 2 f64: BasicOpponent.phase of the player-1 and player-2 controllers */
  HK_S_EPISODE = 48,  /* u32 episodes started (RNG counter for reset draws) */
  HK_S_TICK = 49,     /* u32 ticks executed since creation (RNG counter for per-tick draws) */
  HK_S_RET = 50,      /* 2 f64: running episode return of player 1 and player 2 (statistics only) */
  HK_S_PUCK_C0 = 54,  /* 2 f32: b2Sweep::c0 of the puck (only read if the puck is woken mid-step while asleep) */
  HK_S_MODE = 56,     /* u32 mode of the running episode: 0 = the handle's creation mode (hk_create), m + 1 = mode m.
                         hk_get_state writes 0 whenever the env plays the creation mode (so the records of single-mode
                         handles do not depend on this word); hk_set_state reads 0 and any value above 3 as the creation
                         mode.  Words 57-63 are unused (0). */
  HK_S_CONTACT = 64,  /* HK_N_PAIRS records of HK_CONTACT_WORDS words */
  HK_N_PAIRS = 27,
  HK_CONTACT_WORDS = 8,
  HK_STATE_WORDS = 64 + 27 * 8
};
/* contact record: word0 = flags (bit0 exists, bit1 touching, bits8-15 position in the world contact
 * list, 0 = head/newest); word1 = manifold pointCount; word2,3 = b2ContactID keys; word4,5 = normal,
 * tangent impulse of point 0; word6,7 = of point 1.
 * Pair ids: 0-7 racket1 x {wall top, bottom, left-top, left-bottom, right-top, right-bottom,
 * goal1 solid, goal2 solid}; 8-15 racket2 x same; 16 racket1 x racket2; 17-22 puck x walls;
 * 23,24 puck x goal1/goal2 sensor; 25,26 puck x racket1/racket2. */

/* ---- lifecycle ------------------------------------------------------------------------------ */
/* Replaces HockeyEnv.__init__ (hockey_env.py:91-155) for n_envs envs on CUDA device `device`.
 * env_id_offset: global id of env 0 (RNG streams are keyed on global ids so that results do not
 * depend on how a batch is sharded over GPUs).  Every env starts reset with one_starting = true. */
int hk_create(hk_env** out, int64_t n_envs, int mode, int keep_mode, int device, uint64_t seed,
              int64_t env_id_offset);
int hk_destroy(hk_env* env);
int64_t hk_num_envs(const hk_env* env);

/* Replaces HockeyEnv.reset (hockey_env.py:345-418).  mask_dev: n_envs bytes, nonzero = reset that
 * env (NULL = all).  one_starting_dev: n_envs int8, 1/0 = forced side, -1 = alternate as the
 * reference does when one_starting is None (hockey_env.py:359-362) (NULL = alternate).
 * obs_dev [n,18] f32 (nullable) receives the post-reset observation. */
int hk_reset(hk_env* env, const uint8_t* mask_dev, const int8_t* one_starting_dev, float* obs_dev, void* stream);
/* HockeyEnv.reset(seed=...) (hockey_env.py:347 `self.seed(seed)`: the reference reseeds its generator on every reset, so
 * the reset draws are a function of the seed alone; rl/utils/evaluator.py:18 relies on it with seed = agent.seed + i).
 * seeds_dev: n_envs int64 (nullable); seeds_dev[i] >= 0 = that env's reset draws come from Philox keyed on this seed only
 * (same seed -> same start state on any env of any batch); < 0 = the env's own stream as in hk_reset. */
int hk_reset_seeded(hk_env* env, const uint8_t* mask_dev, const int8_t* one_starting_dev, const int64_t* seeds_dev,
                    float* obs_dev, void* stream);

/* Replaces HockeyEnv.step / HockeyEnv_BasicOpponent.step (hockey_env.py:658-695, :882-886).
 * action_dev: f32 [n, action_stride]; player 1 reads columns 0..3 when p1_policy is EXTERNAL,
 * player 2 reads columns 4..7 when p2_policy is EXTERNAL (needs action_stride >= 8).  May be NULL
 * when neither policy is EXTERNAL.
 * Outputs (all nullable except obs_dev): obs [n,18] f32; obs2 = obs_agent_two() [n,18];
 * reward / reward2 [n] f32 (get_reward / get_reward_agent_two); done [n] u8; info / info2 [n,4] f32
 * (_get_info / get_info_agent_two); final_obs [n,18] (terminal obs when autoreset). */
int hk_step(hk_env* env, const float* action_dev, int action_stride, int p1_policy, int p2_policy, int flags,
            float* obs_dev, float* obs2_dev, float* reward_dev, float* reward2_dev, uint8_t* done_dev,
            float* info_dev, float* info2_dev, float* final_obs_dev, void* stream);

/* One tick for a HOST-side agent (the reference's own calling pattern: numpy in, numpy out).  action_host: PINNED host
 * memory, f32 [n, action_stride] (nullable when no policy is EXTERNAL); record_host: PINNED host memory of
 * hk_host_record_bytes(n, with_final_obs, offsets) bytes laid out as obs [n,18] f32 | reward [n] f32 | info [n,4] f32 |
 * done [n] u8 (| final_obs [n,18] f32) at offsets[0..4]; action_dev / record_dev: caller-owned device scratch of the same
 * sizes.  The actions are copied in on `stream`, the fast tier writes its rows to the device record, a copy engine moves
 * that record to the host on an internal side stream WHILE the general tier runs, and the general tier stores its own
 * rows straight into the mapped host record once that copy has landed -- so almost all of the device-to-host traffic
 * overlaps the tick.  Everything is ordered into `stream`: after a synchronize on it the host record holds the tick's
 * results.  Not CUDA-graph capturable. */
int64_t hk_host_record_bytes(int64_t n_envs, int with_final_obs, int64_t* offsets5);
int hk_step_host(hk_env* env, const float* action_host, int action_stride, int p1_policy, int p2_policy, int flags,
                 float* action_dev, uint8_t* record_dev, uint8_t* record_host, int with_final_obs, void* stream);

/* Per-env opponent selection (the reference draws an opponent per episode from a pool: weak / strong
 * BasicOpponent or a self-play snapshot, rl/training/opponent_manager.py:62-91, rl/training/self_play.py:7-68).
 * codes_dev: n_envs bytes of HK_POLICY_EXTERNAL..HK_POLICY_ZERO, caller-owned device memory that must stay valid
 * while p2_policy == HK_POLICY_PER_ENV is in use (it is read by every such hk_step; the caller may rewrite it
 * between steps, e.g. for the envs that just finished an episode).  EXTERNAL envs read columns 4..7 of action_dev
 * (a snapshot actor's output on obs_agent_two()); the others run their in-kernel controller.  NULL clears it. */
int hk_set_opponent_policies(hk_env* env, const uint8_t* codes_dev);

/* Per-env game mode (the reference's `mode` setter and reset(mode=...), hockey_env.py:345-364, 754-779: the mode of an
 * env is read at each reset and sets the start layout, max_timesteps 250 / 80 and with it the reward scales).
 * modes_dev: n_envs bytes of HK_MODE_NORMAL..HK_MODE_TRAIN_DEFENSE, caller-owned device memory that must stay valid while
 * it is set.  Every later reset of an env -- hk_reset / hk_reset_seeded (masked) and the auto-reset of hk_step /
 * hk_step_host / hk_rollout -- reads its byte and starts the next episode in that mode; the caller may rewrite it between
 * calls (e.g. curriculum draws for the envs that just finished).  The contents are validated once, here.  NULL clears it:
 * each env then keeps the mode it has (every env of a new handle plays the creation mode of hk_create). */
int hk_set_reset_modes(hk_env* env, const uint8_t* modes_dev);
/* The mode of each env's running episode: modes_dev [n] u8.  Asynchronous on `stream`; graph-capturable. */
int hk_get_modes(hk_env* env, uint8_t* modes_dev, void* stream);

/* k_steps ticks with in-kernel policies (no EXTERNAL), autoreset on, enqueued back to back without any
 * per-tick output: only the last tick's obs (nullable) is written; episode statistics accumulate in
 * the handle (hk_get_stats).  (With HK_MONO=1 the k_steps ticks are fused into ONE launch with the
 * body state held in registers between ticks.) */
int hk_rollout(hk_env* env, int k_steps, int p1_policy, int p2_policy, float* obs_dev, void* stream);

/* Observations of the current state without stepping (_get_obs / obs_agent_two, hockey_env.py:485-516). */
int hk_get_obs(hk_env* env, float* obs_dev, float* obs2_dev, void* stream);

/* _get_info / get_info_agent_two of the current state without stepping (what reset() returns,
 * hockey_env.py:416-418, 542-591).  info_dev / info2_dev: f32 [n,4], nullable. */
int hk_get_info(hk_env* env, float* info_dev, float* info2_dev, void* stream);

/* Superset of HockeyEnv.set_state (hockey_env.py:594-608): the full record incl. hidden state. */
int hk_get_state(hk_env* env, uint32_t* state_dev /* [n, HK_STATE_WORDS] */, void* stream);
int hk_set_state(hk_env* env, const uint32_t* state_dev, void* stream);
/* Exactly HockeyEnv.set_state: inject the 18 visible values (f32 [n,18]); hidden state untouched. */
int hk_set_obs_state(hk_env* env, const float* obs18_dev, void* stream);

/* Episode statistics accumulated on the device since creation / last hk_clear_stats.
 * out_host[HK_STATS_DIM] doubles: 0 episodes, 1 wins(+1), 2 losses(-1), 3 draws, 4 env-steps,
 * 5 sum return p1, 6 sum return p2, 7 sum return^2 p1, 8 sum episode length, 9 puck touches p1,
 * 10 puck touches p2, 11 velocity-solver iterations executed, 12 TOI events, 13 contact-list
 * overflows (must be 0), 14 env-steps completed by the general tier(s) (the rest finished in the fast / touch tier),
 * 15 reserved.  Synchronises `stream`. */
int hk_get_stats(hk_env* env, double* out_host, void* stream);
int hk_clear_stats(hk_env* env, void* stream);
/* Device pointer to HK_STATS_DIM doubles holding the accumulators as of this call (summed on the legacy default stream
 * from the library's replicated per-block rows), for an NCCL all-reduce without a host hop. */
int hk_stats_device_ptr(hk_env* env, double** out_dev);
/* Device-to-device copy of the accumulators into a caller-owned f64[HK_STATS_DIM] buffer (async). */
int hk_copy_stats(hk_env* env, double* dst_dev, void* stream);

/* Diagnostics: block-cycles the general tiers spent in each tick phase since creation (synchronises the device).
 * out_host8 = tier 1 {policy+Collide, island solve, TOI, finish}, tier 2 {same}. */
int hk_debug_phase_cycles(hk_env* env, double* out_host8);
/* Diagnostics: block-cycles of the general tier's finish phase as warp 0 of each block saw them: {wait after the TOI
 * barrier, cache commit, tickFinish (info / reward / outputs / auto-reset), state store, statistics flush, final barrier}. */
int hk_debug_finish_cycles(hk_env* env, double* out_host6);
/* Diagnostics (env created with HK_LANE_TRACE=1 in the environment): the last tick's general-tier trace,
 * [n/32+8 warps][4] cycles per tick phase of each warp, then [n][2] per-env work record (hk_lib.cu). */
int hk_debug_lane_trace(hk_env* env, uint32_t* out_host, int64_t n_words);
/* Kernels one hk_step launches on this handle (k_fast, k_touch, general tier(s)); for launch accounting. */
int hk_launches_per_step(const hk_env* env);

/* The reference's TD3 actor (ActorNetwork.forward, rl/td3/networks.py:17-20: 18 -> 256 -> 256 -> 4, tanh after every layer)
 * as one fused tensor-core kernel (BASELINE config 5): act[i, 0..3] = actor(obs[i, 0..17]) for n rows.  params_dev: the
 * hk_actor_param_bytes()-byte block laid out as csrc/hk_actor.cuh describes (bf16 weights in UMMA core-matrix order, f32
 * biases; hockey_env_b200.actor.FusedActor packs it from a torch module).  obs_dev: f32 [n, 18] contiguous; act_dev: f32
 * rows of act_stride >= 4 floats (e.g. the [n, 4] or [n, 8] action tensor of the next hk_step).  bf16 operands, fp32
 * accumulation.  Enqueued on `stream`; graph-capturable. */
int hk_actor_param_bytes(void);
int hk_actor_forward(const void* params_dev, const float* obs_dev, float* act_dev, int act_stride, int64_t n, int device,
                     void* stream);

/* Snapshot pool of the same actor (self-play opponents, league play): act[i, 0..3] = actor_{choice[i]}(obs[i, 0..17]) for
 * every row with 0 <= choice[i] < k; rows with any other choice (negative included) are NOT written.  params_dev: k
 * hk_actor_param_bytes()-byte blocks back to back (snapshot s at s * hk_actor_param_bytes(); 16-byte aligned).
 * choice_dev: i32 [n] (4-byte aligned); obs_dev / act_dev / act_stride as for hk_actor_forward; 1 <= n <= 2^31 - 1,
 * 1 <= k <= 4096.  scratch_dev: caller-owned device memory of hk_actor_pool_scratch_bytes(n, k) bytes (16-byte aligned,
 * contents need not be initialised; one call at a time per buffer); the library allocates nothing per call.
 * Each output row equals hk_actor_forward of its snapshot on that row, bit for bit.  The rows are grouped by snapshot
 * on the device (a memset and three small kernels: histogram, offsets, row lists), then one persistent tensor-core
 * kernel runs tiles of 128 rows of one snapshot each, copying a snapshot's weights into shared memory when its tiles
 * start.  Enqueued on `stream` with no host synchronisation; graph-capturable.  Invalid arguments return HK_E_INVALID
 * (before any device probe); valid ones without a GPU HK_E_NODEVICE.
 * hk_actor_pool_scratch_bytes returns HK_E_INVALID for n or k out of range. */
int64_t hk_actor_pool_scratch_bytes(int64_t n, int k);
int hk_actor_forward_pool(const void* params_dev, int k, const int32_t* choice_dev, const float* obs_dev, float* act_dev,
                          int act_stride, int64_t n, void* scratch_dev, int device, void* stream);

/* The same two kernels with Gaussian noise in the output epilogue (TD3 exploration, target-policy smoothing):
 * act[i] = clamp(tanh(MLP(obs[i])) + c(sigma * z_i), -1, 1), c = clip to [-clip, clip] (clip <= 0 or +inf: no clip).
 * z_i: four standard normals from one Philox4x32-10 call keyed on (seed, row0 + i, *counter_dev) and Box-Muller; the
 * exact key and uniform mapping are in csrc/hk_actor.cuh (NoiseKey).  Row i's noise depends only on that key (not on n,
 * tile order or pool grouping); row0 lets the shards of one batch agree.  counter_dev: one u64 in device memory (8-byte
 * aligned) read by the kernel, so a captured graph draws fresh noise on each replay if the caller advances it.
 * sigma must be finite and >= 0; sigma == 0 gives output bit-identical to hk_actor_forward / hk_actor_forward_pool.
 * Other arguments and error rules as for those two; row0 >= 0.  Enqueued on `stream`; graph-capturable. */
int hk_actor_forward_noisy(const void* params_dev, const float* obs_dev, float* act_dev, int act_stride, int64_t n, uint64_t seed,
                           const uint64_t* counter_dev, float sigma, float clip, int64_t row0, int device, void* stream);
int hk_actor_forward_pool_noisy(const void* params_dev, int k, const int32_t* choice_dev, const float* obs_dev, float* act_dev,
                                int act_stride, int64_t n, void* scratch_dev, uint64_t seed, const uint64_t* counter_dev, float sigma,
                                float clip, int64_t row0, int device, void* stream);

/* Pack an ActorNetwork's fp32 parameters on the device into one hk_actor_param_bytes() block, byte-identical to
 * hockey_env_b200.actor.FusedActor.pack: w1 [256, 18], b1 [256], w2 [256, 256], b2 [256], w3 [4, 256], b3 [4], contiguous
 * f32 device arrays (4-byte aligned).  params_dev: 16-byte aligned; may point into a pool table (slot s at
 * s * hk_actor_param_bytes()) to refresh one snapshot in place.  One small kernel on `stream`, no host synchronisation;
 * graph-capturable.  Invalid arguments return HK_E_INVALID (before any device probe); valid ones without a GPU
 * HK_E_NODEVICE. */
int hk_actor_pack(const float* w1, const float* b1, const float* w2, const float* b2, const float* w3, const float* b3,
                  void* params_dev, int device, void* stream);

/* One TD3 learner update (hockey_env_b200.td3.FusedTD3Learner) in ONE kernel launch: gather, target policy smoothing,
 * twin-critic forward / backward / Adam, prioritized importance weights and priority write-back, and with do_actor the
 * actor forward through the stepped Q1, actor backward / Adam and Polyak of both target nets.  Reference architecture
 * only: actor 18-256-256-4, twin critic 22-256-256-1.  The numerics contract is stated in csrc/hk_td3.cuh.
 *
 * arena_dev: hk_td3_arena_bytes() bytes, 16-byte aligned, fp32 offsets (in floats):
 *   actor params        0        (71,684: fc1.weight [256,18], fc1.bias, fc2.weight [256,256], fc2.bias, fc3.weight [4,256], fc3.bias)
 *   critic params       71,744   (143,874: q1.fc1.weight [256,22], q1.fc1.bias, q1.fc2.*, q1.fc3.weight [1,256], q1.fc3.bias, q2.*)
 *   target actor        215,680, target critic 287,424, Adam m / v of the actor 431,360 / 503,104,
 *   Adam m / v of the critic 574,848 / 718,784,
 *   counters            862,720  (int64: critic step, actor step, target-noise counter)
 * Every net is in state_dict order, row-major as torch stores it; each block starts at a multiple of 64 floats.
 * scratch_dev: hk_td3_scratch_bytes(batch) bytes, 16-byte aligned, contents need not be initialised; its first `batch`
 * floats hold the batch's importance weights after the call.  One call at a time per arena and per scratch buffer.
 * batch->idx: [batch] int64 rows of the replay arrays (each in [0, capacity): not checked).  batch->prio_weights: NULL for
 * a uniform batch; otherwise the buffer's weights, indexed by batch->prio_idx, with N = prio_n >= 1.
 * losses_dev: [2] floats, actor loss (written on actor steps only) and critic loss.
 * Enqueued on `stream` with no host synchronisation and no allocation; graph-capturable.  Invalid arguments (NULL
 * pointers, misalignment, batch outside [1, 1024], non-finite or negative lr / tau / gamma / sigma / clip / wd / beta,
 * prio_n < 1) return HK_E_INVALID before any device probe; valid ones without a GPU HK_E_NODEVICE.
 * hk_td3_scratch_bytes returns HK_E_INVALID for batch out of range. */
typedef struct {
  const float* obs;          /* [capacity, 18] */
  const float* action;       /* [capacity, 4] */
  const float* reward;       /* [capacity] */
  const float* next_obs;     /* [capacity, 18] */
  const float* done;         /* [capacity], 0 or 1 */
  const int64_t* idx;        /* [batch], 8-byte aligned */
  float* prio_weights;       /* NULL: uniform batch */
  const int64_t* prio_idx;   /* [batch] (prioritized only) */
  int64_t prio_n;            /* number of stored transitions (prioritized only) */
} hk_td3_batch;
typedef struct {
  float gamma, tau_actor, tau_critic, lr_actor, lr_critic, wd_actor, wd_critic, beta;
  float target_noise, target_noise_clip;
} hk_td3_hparams;
int64_t hk_td3_arena_bytes(void);
int64_t hk_td3_scratch_bytes(int batch);
int hk_td3_update(void* arena_dev, void* scratch_dev, const hk_td3_batch* batch, int batch_size, const hk_td3_hparams* hp,
                  const float* action_low_dev, const float* action_range_dev, uint64_t seed, int do_actor, float* losses_dev,
                  int device, void* stream);
/* The cluster size (CTAs) that hk_td3_update launches with on `device`: 16 when the device can co-schedule such a
 * cluster, else 8, or lower when the environment variable HK_TD3_CLUSTER (read once per process) asks for a smaller
 * size >= 1.  Results do not depend on it.  HK_E_NODEVICE without a GPU, HK_E_INVALID for a bad device index. */
int hk_td3_cluster_size(int device);

/* K independent TD3 learners (a seed or hyper-parameter sweep, population-based training) updated in ONE launch of K
 * clusters: cluster m runs exactly hk_td3_update's update for member m, so the result of every member is byte-identical
 * to an hk_td3_update call with member m's arguments (the single-member oracle).  1 <= k <= HK_TD3_MAX_POPULATION.
 * Per member m:
 *   arena      arenas_dev + m * hk_td3_arena_bytes() (K arenas back to back);
 *   scratch    scratch_dev + m * hk_td3_scratch_bytes(batch_size) (its first batch_size floats: member m's importance
 *              weights after the call);
 *   indices    batch->idx + m * batch_size, and for a prioritized batch batch->prio_idx + m * batch_size ([k][batch] int64
 *              each, rows of the replay arrays that all members share);
 *   hp[m], seeds[m], do_actor[m] (nonzero: an actor step), action_low[m] / action_range[m] (device pointers to the member
 *   critic's [4] buffers; the two pointer tables are host arrays), losses_dev + 2 * m (actor loss on actor steps only,
 *   critic loss).
 * Shared: the replay arrays, batch_size (1..1024), batch->prio_weights and batch->prio_n (every member's N).  For a
 * prioritized batch, member m's prio_idx must point at rows only member m uses (its own part of the buffer), so that the
 * priority write-backs of different members never overlap; the members' updates are otherwise independent.
 * Everything travels in the launch's parameters (no device-side table, no host-to-device copy, no allocation, no host
 * synchronisation): graph-capturable like hk_td3_update.  Invalid arguments (as for hk_td3_update, plus k outside [1, 64]
 * and NULL or misaligned per-member pointers) return HK_E_INVALID before any device probe, with the member index and the
 * field in the message (e.g. "hk_td3_update_population: member 3: lr_critic must be finite and >= 0"); valid ones
 * without a GPU HK_E_NODEVICE. */
#define HK_TD3_MAX_POPULATION 64
int hk_td3_update_population(void* arenas_dev, void* scratch_dev, const hk_td3_batch* batch, int batch_size, int k,
                             const hk_td3_hparams* hp /* [k] */, const float* const* action_low /* [k] */,
                             const float* const* action_range /* [k] */, const uint64_t* seeds /* [k] */,
                             const uint8_t* do_actor /* [k] */, float* losses_dev /* [k][2] */, int device, void* stream);
/* The cluster size (CTAs per member) of a population launch of k members on `device`: the largest of {16, 8} at which the
 * device keeps all k clusters resident at once (cudaOccupancyMaxActiveClusters >= k), else 16; never above
 * hk_td3_cluster_size(device).  Results do not depend on it.  HK_E_INVALID for k outside [1, 64] or a bad device index,
 * HK_E_NODEVICE without a GPU. */
int hk_td3_population_cluster_size(int k, int device);

/* Repack K actors into K slots of a pool table (hk_actor_forward_pool) in one launch: slot s (at table_dev +
 * s * hk_actor_param_bytes(), 16-byte aligned) is packed from the actor whose fp32 parameters lie back to back in
 * state_dict order (fc1.weight [256,18], fc1.bias, fc2.weight [256,256], fc2.bias, fc3.weight [4,256], fc3.bias) at
 * actors_dev + s * stride_floats (4-byte aligned; stride_floats >= 71,684).  That is the actor block of a TD3 arena, so
 * actors_dev = the first arena and stride_floats = hk_td3_arena_bytes() / 4 repack a whole population.  Each slot is
 * byte-identical to hk_actor_pack of the same actor; slots >= k are not touched.  1 <= k <= 4096.  Error rules and
 * stream semantics as for hk_actor_pack. */
int hk_actor_pack_many(const float* actors_dev, int64_t stride_floats, int k, void* table_dev, int device, void* stream);

/* Measurement: per-kernel device times of the ticks that follow.  hk_kernel_timing(env, 1) makes every hk_step /
 * hk_rollout tick record CUDA events on the launching stream around each kernel of the cascade (up to 2048 ticks; not
 * graph-capturable while enabled); hk_kernel_times synchronises the device, returns the summed milliseconds of
 * {k_fast, k_touch, general tier, second general tier} and the number of ticks they cover, and restarts the record. */
int hk_kernel_timing(hk_env* env, int enable);
int hk_kernel_times(hk_env* env, double* out_ms4, int64_t* steps_out);

const char* hk_last_error(void);
const char* hk_version(void);

#ifdef __cplusplus
}
#endif
#endif /* HOCKEY_B200_H */
