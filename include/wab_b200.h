/*
 * wab_b200.h — C ABI of the B200-native batched Wolves-and-Bushes simulator.
 *
 * The reference (johnmatthewtennant/wab-gym) has no FFI / plugin layer: its only boundary is the
 * Python gym surface of WolvesAndBushesEnv (/root/reference/wab_env.py:103-342). This header is the
 * boundary a binding for that surface calls into; each entry point names the reference interface it
 * replaces. Plain pointers and sizes only — no torch types. All `d_*` pointers are DEVICE pointers
 * owned by the caller (16-byte aligned for `d_grids`), all work is enqueued on the caller's
 * cudaStream_t (passed as void* so C callers need no CUDA headers), nothing synchronises unless
 * stated. One handle <-> one device <-> one stream at a time; handles are independent.
 *
 * Return value of every int function: 0 on success, a WAB_E_* code otherwise; the message is
 * available from wab_last_error() (thread-local).
 */
#ifndef WAB_B200_H
#define WAB_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WAB_ABI_VERSION 1
#define WAB_MAX_ACTIONS 8

enum {
    WAB_OK = 0,
    WAB_E_NULL = 1,        /* null pointer argument                                              */
    WAB_E_CONFIG = 2,      /* invalid option values (reference: ValueError, wab_env.py:147-148)  */
    WAB_E_UNSUPPORTED = 3, /* valid for the reference but outside what the kernels implement     */
    WAB_E_CUDA = 4,        /* CUDA runtime error (message carries cudaGetErrorString)            */
    WAB_E_NO_DEVICE = 5    /* no CUDA device: there is no CPU fallback                           */
};

/* Food arithmetic. The reference keeps food as float64 (wab_env.py:307-322, :452). WAB_FOOD_INT is
 * an integer counter in units of 1/turns_to_empty_food, legal only when the host has proven it
 * equivalent for every reachable state (wab_gym_b200/config.py: prove_integer_food). */
enum { WAB_FOOD_F64 = 0, WAB_FOOD_INT = 1 };

/* Rule constants — the POD image of `default_game_options` (wab_env.py:11-39) plus the action table
 * (wab_env.py:149-182) and host-precomputed integer thresholds for the keyed draws. */
typedef struct WabConfig {
    int32_t abi_version;          /* WAB_ABI_VERSION                                               */
    int32_t width, height;        /* viewport (odd; kernels implement 11x11)      wab_env.py:25-26 */
    int32_t max_turns;            /*                                              wab_env.py:23    */
    int32_t wolf_spawn_margin;    /* kernels implement 1                          wab_env.py:34    */
    int32_t n_actions;            /* 5 or 6                                       wab_env.py:149-191 */
    int8_t action_dx[WAB_MAX_ACTIONS];
    int8_t action_dy[WAB_MAX_ACTIONS];
    int8_t action_role[WAB_MAX_ACTIONS]; /* -1 = keep role (NaN in the reference) wab_env.py:257-258 */
    uint8_t lookout_only;         /*                                              wab_env.py:19, :302 */
    uint8_t restrict_view;        /*                                              wab_env.py:20, :351 */
    uint8_t wolves;               /*                                              wab_env.py:37    */
    uint8_t wolves_can_move;      /*                                              wab_env.py:38    */
    uint8_t god_mode;             /*                                              wab_env.py:292   */
    int8_t starting_role;         /* -1 = random                                  wab_env.py:598-599 */
    uint8_t food_mode;            /* WAB_FOOD_F64 / WAB_FOOD_INT                                   */
    uint8_t auto_reset;           /* 1: done envs are reset inside step() and their post-reset
                                     observation is returned (VecEnv); 0: reference behaviour,
                                     stepping after done keeps returning done     wab_env.py:328-340 */
    int32_t food_int_start;       /* INT mode: starting_food * turns_to_empty_food                 */
    int32_t food_int_inc;         /* INT mode: turns_to_empty_food / turns_to_fill_food            */
    int32_t food_int_max;         /* INT mode: turns_to_empty_food (clip upper bound)              */
    int32_t wolf_cap;             /* wolf slots per env (<= 64); overflow is counted, see stats    */
    int32_t log_cap;              /* depletion-log slots per env (<= 255); overflow is counted     */
    double food_start;            /* F64 mode: starting_food; < 0 = random        wab_env.py:596-597 */
    double food_inc;              /* 1 / turns_to_fill_food                       wab_env.py:307-309 */
    double food_dec;              /* 1 / turns_to_empty_food                      wab_env.py:316   */
    double food_obs_scale;        /* turns_to_empty_food                          wab_env.py:452   */
    /* binomial-first draws (oracle/keyed_rng.py): K = #{k < 32 : v >= cdf[k]} events among n cells, v a 64-bit
       draw; cdf[k] = min(ceil(BinomialCDF(n, chance/2; k) * 2^64), 2^64 - 1)                                  */
    uint64_t spawn_cdf[32];       /* n = 48 ring cells per step                   wab_env.py:571-574 */
    uint64_t init_cdf[32];        /* n = 121 window cells per reset               wab_env.py:588-591 */
    uint64_t thr_keep;            /* wolf kept iff word >= thr (U > despawn)      wab_env.py:262-264 */
    float reward_table[8];        /* [ate*4 + outcome], outcome 0 alive, 1 finished, 2 starved,
                                     3 killed; the f32 image of the fp64 sums     wab_env.py:328-340 */
    uint32_t mask_lookout[4];     /* 121-bit blind-spot masks, bit = i*11 + j     wab_env.py:109-139 */
    uint32_t mask_gatherer[4];
} WabConfig;

/* Observation batch: the first six elements of the reference's tuple (wab_env.py:374-385) for N
 * envs. The seventh (view_mask) is a function of role and options only. */
typedef struct WabObs {
    uint8_t *d_grids;  /* [N][3][11][11] u8: wolves, bushes, ostriches; cell [i][j] = [5-dx][5-dy]. May be NULL in
                        * wab_vec_reset / wab_vec_step / wab_vec_step_many while a feature buffer is bound
                        * (wab_vec_bind_features): FEATURES-ONLY stepping — the 28 PragmaticObsWrapper bytes per env, the
                        * scalars, reward, done and info are written, the one-hot grids are not materialised. */
    uint8_t *d_food;   /* [N] ceil(food * turns_to_empty_food)                     wab_env.py:452  */
    uint8_t *d_role;   /* [N]                                                      wab_env.py:390  */
    uint8_t *d_status; /* [N] 0 alive, 1 starved, 2 killed                         wab_env.py:387  */
} WabObs;

/* info byte written by step (optional): bits 0-1 outcome (index into reward_table), bit 2 ate,
 * bit 3 invalid action, bits 4-5 status before auto-reset. */
#define WAB_INFO_OUTCOME(b) ((b) & 3)
#define WAB_INFO_ATE(b) (((b) >> 2) & 1)
#define WAB_INFO_BAD_ACTION(b) (((b) >> 3) & 1)
#define WAB_INFO_FINAL_STATUS(b) (((b) >> 4) & 3)

/* indices into the int64[8] vector of wab_vec_stats */
enum {
    WAB_STAT_EPISODES = 0, WAB_STAT_STEPS = 1, WAB_STAT_FINISHED = 2, WAB_STAT_STARVED = 3,
    WAB_STAT_KILLED = 4, WAB_STAT_EATS = 5, WAB_STAT_BAD_ACTIONS = 6, WAB_STAT_OVERFLOWS = 7
};

typedef struct WabVec WabVec;

/* Replaces WolvesAndBushesEnv.__init__ (wab_env.py:106-186) for n_envs environments with global ids
 * env_id_base .. env_id_base + n_envs - 1 (keys depend on the global id only, so results do not
 * depend on how a batch is sharded over GPUs). bush_thr[k-1] = least 32-bit draw whose bush value
 * round(U**bush_power * max_berries) is >= k (wab_env.py:631-635). Allocates state on `device`.
 * Does NOT reset (the reference constructor does, :186): call wab_vec_reset. */
int wab_vec_create(const WabConfig *cfg, const uint32_t *bush_thr, int32_t n_bush_thr, int64_t n_envs,
                   uint64_t seed, uint64_t env_id_base, int32_t device, WabVec **out);

/* Replaces reset() (wab_env.py:231-248). d_mask: NULL = all envs, else u8[N], nonzero = reset. Each
 * reset env starts its next episode (first reset -> episode 0). Observations are written for EVERY
 * env: the others get the observation their last step returned again — including the bush under the
 * ostrich if that step ate it empty, which the reference's observation still shows because its frame
 * (wab_env.py:266) predates the eat (:300-313) and is only rebuilt by the next step. */
int wab_vec_reset(WabVec *h, const uint8_t *d_mask, WabObs obs, void *stream);

/* Replaces step(action) (wab_env.py:250-342) for all envs. d_actions u8[N]; outputs: obs, d_reward
 * f32[N], d_done u8[N], d_info u8[N] (may be NULL). */
int wab_vec_step(WabVec *h, const uint8_t *d_actions, WabObs obs, float *d_reward, uint8_t *d_done,
                 uint8_t *d_info, void *stream);

/* T lockstep steps in ONE launch: d_actions u8[T][N]; every step's results are materialised:
 * grids [T][N][3][11][11], food/role/status/done/info [T][N], reward [T][N] (info may be NULL). */
int wab_vec_step_many(WabVec *h, int32_t n_steps, const uint8_t *d_actions, WabObs obs, float *d_reward,
                      uint8_t *d_done, uint8_t *d_info, void *stream);

/* Same contract as wab_vec_step with HOST buffers (pageable or pinned): copies actions in, steps,
 * copies every output back, and synchronises the stream before returning. h_info may be NULL. */
int wab_vec_step_host(WabVec *h, const uint8_t *h_actions, uint8_t *h_grids, uint8_t *h_food,
                      uint8_t *h_role, uint8_t *h_status, float *h_reward, uint8_t *h_done,
                      uint8_t *h_info, void *stream);
/* Same step with ONE contiguous host block for every output (one device-to-host transfer instead of
 * seven): wab_vec_host_block_layout gives the byte offsets of grids, food, role, status, reward,
 * done, info inside the block (each 256-byte aligned) and its total size. With PINNED buffers and a batch
 * of at most 16,384 envs the kernel reads the actions from, and writes the block into, host memory directly
 * (no staging copy); either way the block is complete when the call returns. */
int wab_vec_host_block_layout(const WabVec *h, int64_t *offsets7, int64_t *total_bytes);
int wab_vec_step_host_packed(WabVec *h, const uint8_t *h_actions, uint8_t *h_block, void *stream);
/* The host-buffer entry points remember, by host address, what they resolved for the caller's buffers (the device
 * aliases of pinned memory, the captured copy-step-copy graph). Call this before freeing or unregistering a buffer that
 * was passed to them: a later allocation at the same address must not inherit a stale alias. */
int wab_vec_forget_host_buffers(WabVec *h);
int wab_vec_reset_host(WabVec *h, uint8_t *h_grids, uint8_t *h_food, uint8_t *h_role, uint8_t *h_status,
                       void *stream);

/* Episode statistics accumulated on the device since create (or the last call with clear != 0):
 * copies int64[8] (WAB_STAT_*) to h_out8 and synchronises the stream. d_out8 variant: enqueue a
 * device-to-device copy only (for an NCCL all-reduce by the caller), no sync. */
int wab_vec_stats(WabVec *h, int64_t *h_out8, int32_t clear, void *stream);
int wab_vec_stats_device(WabVec *h, int64_t *d_out8, void *stream);

/* Hidden state for differential tests (synchronises). Any pointer may be NULL.
 * x,y i32[N]; food f64[N] (INT mode: counter / turns_to_empty_food); role,status,turn i32[N];
 * episode i64[N]; n_wolves i32[N]; wolves_xy i32[N][wolf_cap][2]; bush_mask u32[N][4];
 * n_log i32[N]; log i32[N][log_cap][3] (x, y, eats). */
int wab_vec_export_state(WabVec *h, int32_t *x, int32_t *y, double *food, int32_t *role, int32_t *status,
                         int32_t *turn, int64_t *episode, int32_t *n_wolves, int32_t *wolves_xy,
                         uint32_t *bush_mask, int32_t *n_log, int32_t *log_xyc, void *stream);

/* ---- checkpoint / resume / clone. The state of one env is one fixed-size, 16-byte-aligned RECORD (little-endian):
 *
 *   byte  0  u32 format        WAB_STATE_FORMAT
 *         4  u32 flags         bit 0: stale centre bush (the last step ate the bush under the ostrich empty); others 0
 *         8  u64 fingerprint   wab_vec_state_fingerprint of the handle that saved it
 *        16  u64 env_id        global id of the env it was saved from
 *        24  u32 episode       28 u32 turn       32 i32 x        36 i32 y
 *        40  u32 role          44 u32 status     48 u32 food counter (WAB_FOOD_INT; 0 in F64 mode)
 *        52  u32 n_wolves      56 f64 food (WAB_FOOD_F64; 0 in INT mode)
 *        64  u32 bkey[2]       the episode's bush key
 *        72  u32 n_log         76 u32 0
 *        80  u32 window[4]     121-bit bush occupancy of the view (specialised kernels; 0 on the generic ones)
 *        96  u32 wolves[wolf_cap]         x:i16 | y:i16 << 16; slots >= n_wolves are 0
 *            u32 log_cell[log_cap]        depletion log, same packing; slots >= n_log are 0
 *            u8  log_count[log_cap]       eats of each logged bush; slots >= n_log are 0
 *            (0-padded to 4 bytes)
 *            u32 hist[max_turns + 1]      only with wab_vec_enable_ego: position after turn t for 1 <= t <= turn, else 0
 *            (0-padded to 16 bytes)
 *
 * Equal states give byte-equal records. The Bloom signature of the log and the "something was eaten empty" flag are not
 * stored: loading rebuilds them from the log. Draws are keyed by the GLOBAL env id of the slot a record is loaded into,
 * so a record loaded into the slot of its own id continues bit for bit on any shard layout, and one loaded into another
 * slot is a clone: same world, ostrich, wolves and log, future draws keyed by the new id. */
#define WAB_STATE_FORMAT 1
/* Bytes of one record for this handle (depends on wolf_cap, log_cap, max_turns and whether ego is enabled). */
int64_t wab_vec_state_record_bytes(const WabVec *h);
/* 64-bit hash of the validated configuration field values, the bush threshold table, the seed, the kernel kind
 * (wab_vec_kernel_kind) and the ego flag; not of env_id_base or n_envs. Records load only into a matching handle. */
int wab_vec_state_fingerprint(const WabVec *h, uint64_t *out);
/* d_slots i32[n] or NULL (= all N envs, n must be N); d_records u8[n][record_bytes], 16-byte aligned. Record r is the state
 * of slot d_slots[r] (or r). Enqueued on the stream, no synchronisation. */
int wab_vec_save_state(WabVec *h, const int32_t *d_slots, int64_t n, void *d_records, void *stream);
/* Record r goes to slot d_slots[r] (NULL = slot r). obs may be all-NULL: state only, no observation written.
 * Otherwise the observation (and bound features) of EVERY env is written, as after wab_vec_reset with an empty mask.
 * *d_rejected (device int32) = number of records refused (format, fingerprint, n_wolves > wolf_cap, n_log > log_cap,
 * role, status, food counter, turn or flags outside what the kernels maintain, slot out of range); when it is non-zero
 * nothing was written. All-or-nothing without a host synchronisation. With duplicate destination slots one of the
 * duplicates wins, unspecified which. */
int wab_vec_load_state(WabVec *h, const void *d_records, const int32_t *d_slots, int64_t n, WabObs obs,
                       int32_t *d_rejected, void *stream);
/* Overwrite the accumulated statistics (row 0 = h_in8, every other per-warp row zeroed). */
int wab_vec_set_stats(WabVec *h, const int64_t *h_in8, void *stream);

int64_t wab_vec_num_envs(const WabVec *h);
/* Lanes cooperating on one env (1, 4, 8, 16 or 32), chosen at create from the batch size so that a
 * small batch still covers every SM; results do not depend on it. */
int wab_vec_lanes_per_env(const WabVec *h);
/* 1 when a wab_vec_step_many launch of n_steps steps runs as the two-warp pipeline (wab_step_pipe_kernel: one warp of a
 * pair runs the rules, the other publishes observations and scalars), 0 when it runs wab_step_kernel. The pipeline serves
 * lanes-per-env batches of up to 8 rule warps per SM and launches of >= 4 steps; WAB_PIPE=0 / 2 in the environment
 * forces never / always. Results are identical. */
int wab_vec_step_many_pipelined(const WabVec *h, int32_t n_steps);
/* Which kernels serve this handle: 0 = the specialised 11 x 11 / spawn-margin-1 kernels (a 121-bit window sliding in
 * registers), 1 = the warp-per-env kernels for every other odd viewport up to 31 x 31 and margins 1, 2 (wab_generic.cuh;
 * WAB_GENERIC=1 in the environment forces them onto the default geometry, for tests). Results are identical. */
int wab_vec_kernel_kind(const WabVec *h);
void wab_vec_destroy(WabVec *h);

/* ---- next row of the path: the reference's PragmaticObsWrapper (wab_env.py:670-824), the observation
 * its actor-critic actually consumes (actor_critic.py:42, :188). 28 bytes per env:
 * nearest_wolf[4] second_wolf[4] n_wolves[4] nearest_bush[4] second_bush[4] n_bushes[4] (each
 * [up, right, down, left]) standing_on_bush food role status. */
#define WAB_FEATURE_BYTES 28
/* Bind (or unbind with NULL) a device buffer u8[N][28] ([T][N][28] for step_many): every later
 * reset/step also writes the features of the observation it returns, fused into the same kernel. */
int wab_vec_bind_features(WabVec *h, uint8_t *d_features);
/* The same features for an arbitrary observation batch already in HBM (replaces
 * PragmaticObsWrapper.observation, wab_env.py:726-761). */
int wab_pragmatic_features(const uint8_t *d_grids, const uint8_t *d_food, const uint8_t *d_role,
                           const uint8_t *d_status, int64_t n, uint8_t *d_features, void *stream);
/* gym.spaces.flatten of the wrapper observation (actor_critic.py:188): f32[n_rows][wab_vec_flat_dim]
 * one-hot vectors (449 for default options) including the role's view mask. */
int wab_vec_flatten_features(WabVec *h, const uint8_t *d_features, int64_t n_rows, float *d_out, void *stream);
int wab_vec_flat_dim(const WabVec *h);
/* The policy input of actor_critic.py:188-189 in one pass: the same one-hot rows plus noise_scale * U[0,1) per element
 * (the reference adds np.random.rand(...) / 100), written as f32 (out_bf16 = 0) or bf16 (1). The draws are keyed by
 * the handle's seed, the element's column, its row's GLOBAL env id (env_id_base + row) and the 64-bit value at
 * d_counter (device memory, may be NULL = 0), which the caller advances between calls — so a captured CUDA graph gets
 * fresh noise on every replay.
 *
 * Keying contract of the policy entry points: every one that takes a WabVec handle (wab_vec_flatten_features_noisy,
 * wab_policy_affine1, wab_policy_trunk, wab_policy_forward, wab_policy_act, wab_policy_backward, wab_policy_ppo_backward,
 * wab_policy_evaluate, wab_policy_backward_logits and the population calls) keys its noise and its action samples by the global env id env_id_base + row (the row within its step for the backward passes; env_id_base + row % n on a handle with replicas, wab_vec_set_replicas, and the block's id on a blocked handle, wab_vec_set_blocks), so
 * a shard [first, first + count) draws exactly what the unsharded batch draws for rows first .. first + count - 1;
 * outputs stay indexed by the local row. The two handle-less calls, wab_sample_categorical and wab_policy_tail, know no
 * shard and key by the local row. */
int wab_vec_flatten_features_noisy(WabVec *h, const uint8_t *d_features, int64_t n_rows, void *d_out,
                                   int32_t out_bf16, float noise_scale, const uint64_t *d_counter, void *stream);

/* Categorical(probs).sample() of the reference's select_action (actor_critic.py:117-120) for n rows of n_actions <= 8
 * probabilities (f32, or bf16 when probs_bf16 = 1), one u8 action per row, on the device: inverse CDF on one
 * uniform per row keyed by (seed, row, *d_counter) — d_counter as in wab_vec_flatten_features_noisy; row is the LOCAL
 * row (no handle, no shard). */
int wab_sample_categorical(const void *d_probs, int32_t probs_bf16, int64_t n, int32_t n_actions, uint64_t seed,
                           const uint64_t *d_counter, uint8_t *d_actions, void *stream);

/* ---- the reference's egocentric observation family (wab_env.py:637-667, WolvesAndBushesEnvEgoCentric :930-958):
 * for the five squares the ostrich can reach next (up, right, down, left, stay) the proximity
 * clip(max_distance - taxicab distance, 0, max_distance), max_distance = 11, of the nearest wolf and of the nearest
 * bush with food among every cell seen this episode. wab_vec_enable_ego (before the first reset) makes the step
 * kernels keep each episode's position history (4 bytes per env-step); wab_vec_ego_proximities writes
 * d_out10 u8[N][10] = wolves[5], bushes[5] for the state left by the last reset/step. Envs stepped past max_turns
 * without a reset keep only their first max_turns positions. */
int wab_vec_enable_ego(WabVec *h);
int wab_vec_ego_proximities(WabVec *h, uint8_t *d_out10, void *stream);

/* Replicas: the handle's N envs become n_replicas copies of n = N / n_replicas envs. Row r takes the global env id
 * env_id_base + r % n in every draw keyed by the global id: the world draws of the step and reset kernels, the origin id
 * written by wab_vec_save_state, and the noise and action samples of the policy entry points (the backward passes'
 * regenerated noise included). So block k of a replicated handle, driven by an action stream, plays exactly what a handle
 * of n envs at env_id_base plays under that stream: several policies can be scored on the same episodes in one launch.
 * n_replicas = 1 is the unreplicated handle. Like wab_vec_enable_ego, valid only before the first reset (or load);
 * WAB_E_CONFIG for n_replicas < 1, a count that does not divide n_envs, n_envs >= 2^32, or a handle already reset. The
 * state fingerprint is unchanged: a record is valid on either kind of handle, and the slot it is loaded into decides its
 * ids. */
int wab_vec_set_replicas(WabVec *h, int64_t n_replicas);

/* Blocks: the handle's N envs become n_blocks blocks of c = N / n_blocks envs, and row r = k c + j takes the global env id
 * env_id_base + k block_stride + j in every draw keyed by the global id (the same sites as for replicas). So block k,
 * driven by an action stream, plays exactly what a handle of c envs at env_id_base + k block_stride plays: a rank of a
 * data-parallel population holds every member's shard of ids on one handle. block_stride = 0 is wab_vec_set_replicas(h,
 * n_blocks); n_blocks = 1 is the plain handle. Valid only before the first reset (or load); WAB_E_CONFIG for n_blocks < 1,
 * a count that does not divide n_envs, a negative block_stride or 0 < block_stride < N / n_blocks (the blocks' ids would
 * overlap), a layout whose last id lies 2^32 or more past env_id_base ((n_blocks - 1) block_stride + N / n_blocks > 2^32),
 * n_envs >= 2^32, or a handle already reset. The state fingerprint is unchanged. */
int wab_vec_set_blocks(WabVec *h, int64_t n_blocks, int64_t block_stride);

/* The first layer of the reference's Policy on the tensor cores (actor_critic.py:59, :88-90, :188-189), fp32 accuracy:
 * d_out f32[n_rows][128] = leaky_relu(affine1(flatten(obs) + noise_scale * U[0,1))) straight from the 28 feature bytes per
 * row (d_features as in wab_vec_flatten_features) — the 449-wide input is generated inside the kernel, with the SAME keyed
 * noise as wab_vec_flatten_features_noisy for the same *d_counter, and never written to memory. One tcgen05 kernel
 * (bf16 x 3 operand splits, fp32 accumulation in tensor memory; the result equals the fp32 GEMM to rounding).
 * wab_policy_affine1_prepare packs affine1.weight f32[128][in_dim] (in_dim = wab_vec_flat_dim, at most 512) into
 * d_packed (wab_policy_affine1_packed_bytes() bytes, 16-byte aligned) — once per weight update; d_bias f32[128]. */
int64_t wab_policy_affine1_packed_bytes(void);
int wab_policy_affine1_prepare(const float *d_weight, int32_t in_dim, void *d_packed, void *stream);
int wab_policy_affine1(WabVec *h, const uint8_t *d_features, int64_t n_rows, const void *d_packed, const float *d_bias,
                       float noise_scale, float leaky_slope, const uint64_t *d_counter, float *d_out, void *stream);

/* The whole trunk of the reference's Policy.forward (actor_critic.py:88-92) in the same tcgen05 kernel, fp32 accuracy:
 * d_z3 f32[n_rows][128] = affine3(leaky_relu(affine2(leaky_relu(affine1(flatten(obs) + noise))))) — the PRE-activation
 * output of affine3, which is what wab_policy_tail takes. The hidden activations never leave the SM: accumulators ->
 * registers (bias, leaky-ReLU, three-way bf16 split) -> shared memory as the next layer's operand. d_packed1 / d_bias1 as
 * for wab_policy_affine1; d_packed2 = wab_policy_linear_prepare(affine2.weight f32[150][128]), d_packed3 =
 * wab_policy_linear_prepare(affine3.weight f32[128][150]) (wab_policy_linear_packed_bytes(n_out, n_in) bytes each,
 * 16-byte aligned; once per weight update); hidden2 must be 150. */
int64_t wab_policy_linear_packed_bytes(int32_t n_out, int32_t n_in);
int wab_policy_linear_prepare(const float *d_weight, int32_t n_out, int32_t n_in, void *d_packed, void *stream);
int wab_policy_trunk(WabVec *h, const uint8_t *d_features, int64_t n_rows, const void *d_packed1, const float *d_bias1,
                     const void *d_packed2, const float *d_bias2, int32_t hidden2, const void *d_packed3,
                     const float *d_bias3, float noise_scale, float leaky_slope, const uint64_t *d_counter, float *d_z3,
                     void *stream);

/* Policy.forward + select_action (actor_critic.py:84-97, :108-125) for n_rows environments as ONE kernel: wab_policy_trunk
 * followed, in the same launch, by what wab_policy_tail does (x = clamp(leaky_relu(z3), lo, hi), both heads, softmax, one
 * action per row by inverse CDF on a uniform keyed by (sample_seed, env_id_base + row, *d_counter)). Arguments as for those two calls;
 * d_value, d_probs, d_logp and d_z3 may be NULL. */
int wab_policy_forward(WabVec *h, const uint8_t *d_features, int64_t n_rows, const void *d_packed1, const float *d_bias1,
                       const void *d_packed2, const float *d_bias2, int32_t hidden2, const void *d_packed3,
                       const float *d_bias3, const float *d_w_heads, const float *d_b_heads, int32_t n_actions,
                       float noise_scale, float leaky_slope, float clamp_lo, float clamp_hi, uint64_t sample_seed,
                       const uint64_t *d_counter, uint8_t *d_actions, float *d_value, float *d_probs, float *d_logp,
                       float *d_z3, void *stream);

/* The greedy (deterministic) action of the same network, for evaluation: wab_policy_forward without sample_seed. The
 * trunk, clamp, heads and softmax are wab_policy_forward's, and so is the keyed input noise (noise_scale = 0 turns it
 * off); d_actions[row] is the first index of the largest logit (the action head's output before the softmax, bias
 * included), so ties go to the lowest index, as torch.argmax does for finite logits. No action sample is drawn.
 * d_value and d_probs are bit-equal to wab_policy_forward's for the same inputs; d_logp is log(p) of the greedy action,
 * bit-equal to wab_policy_forward's wherever the sampled action is the greedy one. Arguments, NULL rules, alignment and
 * return codes as for wab_policy_forward. */
int wab_policy_act(WabVec *h, const uint8_t *d_features, int64_t n_rows, const void *d_packed1, const float *d_bias1,
                   const void *d_packed2, const float *d_bias2, int32_t hidden2, const void *d_packed3,
                   const float *d_bias3, const float *d_w_heads, const float *d_b_heads, int32_t n_actions,
                   float noise_scale, float leaky_slope, float clamp_lo, float clamp_hi, const uint64_t *d_counter,
                   uint8_t *d_actions, float *d_value, float *d_probs, float *d_logp, float *d_z3, void *stream);

/* The backward pass of Policy.forward for training (actor_critic.py:128-169) on the tensor cores. For T = n_steps steps of
 * N = n_envs environments, rows t N + n in step-major order:
 *   d_features u8[T][N][28] (as wab_vec_flatten_features), d_counters int64[T] (the *d_counter each step's
 *   wab_policy_forward saw), d_actions u8[T N], d_g_logp / d_g_value f32[T N] (upstream gradients of the sampled
 *   action's log-probability and of the value).
 * Writes d_grad f32 = the gradient of sum_rows g_logp log pi(a | x) + g_value V(x) in
 * torch.nn.utils.parameters_to_vector(policy.parameters()) order: affine1.weight [128][flat_dim], affine1.bias [128],
 * affine2.weight [150][128], affine2.bias [150], affine3.weight [128][150], affine3.bias [128], action_head.weight [A][128],
 * action_head.bias [A], value_head.weight [1][128], value_head.bias [1].
 * x is the input the forward saw: row n of step t under counter d_counters[t] (the noise key is the global env id
 * env_id_base + n, as wab_vec_flatten_features_noisy / wab_policy_forward key it). The forward is recomputed with wab_policy_forward's
 * arithmetic: d_logp / d_value f32[T N] (each may be NULL) receive the recomputed log pi(a | x) and V(x), bit-identical
 * to what wab_policy_forward returned for the same inputs. d_rows int32[...] / d_n_rows int64[1] (both NULL: every row)
 * restrict the work to the first *d_n_rows entries of d_rows (d_rows must hold that many); the count is read on the device,
 * so the call never synchronises, and is clamped to [0, T N]. Rows left out contribute nothing, as do listed entries
 * outside [0, T N) and rows with zero upstream gradients.
 * d_packed1..3, d_bias1..3, hidden2 (150), d_w_heads / d_b_heads (stacked as for wab_policy_forward) as for
 * wab_policy_forward; d_packed2t = wab_policy_linear_prepare(affine2.weight^T f32[128][150], 128, 150), d_packed3t =
 * wab_policy_linear_prepare(affine3.weight^T f32[150][128], 150, 128). d_scratch: at least
 * wab_policy_backward_scratch_bytes(h) bytes, 16-byte aligned, contents irrelevant. Equal inputs give bit-identical
 * d_grad (fixed-order reductions, no atomics). WAB_E_NULL for a missing pointer, WAB_E_CONFIG for misalignment or too
 * small a scratch, WAB_E_UNSUPPORTED beyond 8 actions, for hidden2 != 150 or flat_dim > 512. */
int64_t wab_policy_backward_scratch_bytes(const WabVec *h);
int wab_policy_backward(WabVec *h, const uint8_t *d_features, int64_t n_steps, int64_t n_envs, const uint64_t *d_counters,
                        const uint8_t *d_actions, const float *d_g_logp, const float *d_g_value, const int32_t *d_rows,
                        const int64_t *d_n_rows, const void *d_packed1, const float *d_bias1, const void *d_packed2,
                        const float *d_bias2, int32_t hidden2, const void *d_packed3, const float *d_bias3,
                        const void *d_packed2t, const void *d_packed3t, const float *d_w_heads, const float *d_b_heads,
                        int32_t n_actions, float noise_scale, float leaky_slope, float clamp_lo, float clamp_hi,
                        void *d_scratch, int64_t scratch_bytes, float *d_grad, float *d_logp, float *d_value, void *stream);

/* PPO's clipped objective through the same backward pass, in one launch per minibatch. Arguments as for
 * wab_policy_backward, except that the upstream gradients are formed on the device from d_logp_old, d_advantage and
 * d_target f32[T N] (the log-probability the action was sampled with, the advantage A, the value target R). d_grad
 * receives the gradient of sum over the listed rows of
 *   l = -policy_weight * min(r A, clip(r, 1 - clip_eps, 1 + clip_eps) A) + value_weight * (V - R)^2 / 2
 *       - entropy_weight * H,
 *   r = exp(log pi(a | x) - logp_old),   H = -sum_o p_o log p_o,
 * with log pi(a | x), V(x) and p recomputed under the current weights (bit-identical to wab_policy_forward's). So
 * g_logp = -policy_weight A r, or 0 where the clip is active (A > 0 and r > 1 + clip_eps, or A < 0 and r < 1 - clip_eps),
 * g_value = value_weight (V - R), and the entropy term adds entropy_weight p_o (log p_o + H) to d logit_o. With the
 * per-row means of a minibatch of M rows, pass weights divided by M. d_logp, d_value and d_entropy f32[T N] (each may be
 * NULL) receive the new log pi(a | x), V(x) and H of the listed rows. WAB_E_NULL for a missing d_logp_old, d_advantage or
 * d_target; WAB_E_CONFIG for clip_eps <= 0 or NaN (+inf disables clipping) or a non-finite weight; otherwise as
 * wab_policy_backward. */
int wab_policy_ppo_backward(WabVec *h, const uint8_t *d_features, int64_t n_steps, int64_t n_envs,
                            const uint64_t *d_counters, const uint8_t *d_actions, const float *d_logp_old,
                            const float *d_advantage, const float *d_target, const int32_t *d_rows, const int64_t *d_n_rows,
                            const void *d_packed1, const float *d_bias1, const void *d_packed2, const float *d_bias2,
                            int32_t hidden2, const void *d_packed3, const float *d_bias3, const void *d_packed2t,
                            const void *d_packed3t, const float *d_w_heads, const float *d_b_heads, int32_t n_actions,
                            float noise_scale, float leaky_slope, float clamp_lo, float clamp_hi, float clip_eps,
                            float policy_weight, float value_weight, float entropy_weight, void *d_scratch,
                            int64_t scratch_bytes, float *d_grad, float *d_logp, float *d_value, float *d_entropy,
                            void *stream);

/* A population of P = n_members policies of the reference's network, 1 <= P <= 64, trained side by side on one handle:
 * member m owns rows [m n, (m + 1) n) of every step, n = member_rows (forward) or n_envs / P (backward), a positive
 * multiple of 128 (a tile of the kernels never straddles two members). Member m's weights are stacked at fixed strides:
 * d_packed1 [P][wab_policy_affine1_packed_bytes()], d_packed2 / d_packed3 / d_packed2t / d_packed3t
 * [P][wab_policy_linear_packed_bytes(..)] of the single-policy layouts, d_bias1 f32[P][128], d_bias2 f32[P][150], d_bias3
 * f32[P][128], d_w_heads f32[P][A + 1][128], d_b_heads f32[P][A + 1]. Every draw is keyed as for one policy (global env id
 * env_id_base + row), so with env_id_base = 0 member m's outputs equal, bit for bit, those of the single-policy call with
 * member m's weights on a handle whose env_id_base is m n.
 *
 * wab_policy_forward_population: wab_policy_forward over P n rows, each row under its member's weights. Arguments, NULL
 * rules and alignment as for wab_policy_forward; WAB_E_CONFIG for P outside [1, 64] or member_rows not a positive
 * multiple of 128, otherwise as wab_policy_forward. wab_policy_act_population is the same call with wab_policy_act's
 * greedy action (no sample_seed), with the same checks and return codes: on a handle with wab_vec_set_replicas(h, P)
 * every member acts on the same envs, which scores P policies on the same episodes in one launch per step.
 *
 * wab_policy_ppo_backward_population: wab_policy_ppo_backward for every member in one launch of P x (the single-policy
 * grid) CTAs. d_rows int32[P][list_len] holds each member's row list as GLOBAL rows t N + n (N = n_envs), d_counts
 * int64[P] the count of each (read on the device, clamped to [0, min(T N, list_len)]); an entry outside [0, T N) or whose
 * env is not in the member's block contributes nothing. h_coefs f32[P][4] (host memory, read during the call):
 * clip_eps, policy_weight, value_weight, entropy_weight of each member, validated as wab_policy_ppo_backward's scalars.
 * d_logp_old, d_advantage, d_target and the optional d_logp, d_value, d_entropy are f32[T N], indexed by global row.
 * Member m's tiles go to its CTAs in the order a single-policy launch uses, so row m of d_grad f32[P][stride], stride =
 * wab_policy_population_grad_stride(h, A) (the parameter count rounded up to 64 floats: with d_grad 256-byte aligned,
 * each member's row is too), equals member m's wab_policy_ppo_backward gradient bit for bit. d_scratch: at least
 * wab_policy_backward_population_scratch_bytes(h, P) = P wab_policy_backward_scratch_bytes(h) bytes (0 for P outside
 * [1, 64]), 16-byte aligned. WAB_E_NULL for a missing d_rows, d_counts, h_coefs or array; WAB_E_CONFIG for P outside
 * [1, 64], n_envs / P not a positive multiple of 128, list_len < 0, a bad coefficient, misalignment or too small a
 * scratch; otherwise as wab_policy_ppo_backward. wab_policy_population_grad_stride returns 0 beyond 8 actions. */
int wab_policy_forward_population(WabVec *h, const uint8_t *d_features, int32_t n_members, int64_t member_rows,
                                  const void *d_packed1, const float *d_bias1, const void *d_packed2, const float *d_bias2,
                                  int32_t hidden2, const void *d_packed3, const float *d_bias3, const float *d_w_heads,
                                  const float *d_b_heads, int32_t n_actions, float noise_scale, float leaky_slope,
                                  float clamp_lo, float clamp_hi, uint64_t sample_seed, const uint64_t *d_counter,
                                  uint8_t *d_actions, float *d_value, float *d_probs, float *d_logp, float *d_z3,
                                  void *stream);
int wab_policy_act_population(WabVec *h, const uint8_t *d_features, int32_t n_members, int64_t member_rows,
                              const void *d_packed1, const float *d_bias1, const void *d_packed2, const float *d_bias2,
                              int32_t hidden2, const void *d_packed3, const float *d_bias3, const float *d_w_heads,
                              const float *d_b_heads, int32_t n_actions, float noise_scale, float leaky_slope,
                              float clamp_lo, float clamp_hi, const uint64_t *d_counter, uint8_t *d_actions,
                              float *d_value, float *d_probs, float *d_logp, float *d_z3, void *stream);
int64_t wab_policy_backward_population_scratch_bytes(const WabVec *h, int32_t n_members);
int64_t wab_policy_population_grad_stride(const WabVec *h, int32_t n_actions);
int wab_policy_ppo_backward_population(WabVec *h, const uint8_t *d_features, int64_t n_steps, int64_t n_envs,
                                       int32_t n_members, const uint64_t *d_counters, const uint8_t *d_actions,
                                       const float *d_logp_old, const float *d_advantage, const float *d_target,
                                       const int32_t *d_rows, int64_t list_len, const int64_t *d_counts,
                                       const void *d_packed1, const float *d_bias1, const void *d_packed2,
                                       const float *d_bias2, int32_t hidden2, const void *d_packed3, const float *d_bias3,
                                       const void *d_packed2t, const void *d_packed3t, const float *d_w_heads,
                                       const float *d_b_heads, int32_t n_actions, float noise_scale, float leaky_slope,
                                       float clamp_lo, float clamp_hi, const float *h_coefs, void *d_scratch,
                                       int64_t scratch_bytes, float *d_grad, float *d_logp, float *d_value,
                                       float *d_entropy, void *stream);

/* Any loss over the policy's outputs: the recomputed forward and the vector-Jacobian product of (logits, value), so a
 * caller can write the loss in torch (or anything else) and keep only the outputs per row, never the activations.
 * Both calls take a LIST of n_rows = M entries: d_rows int32[M] (device; NULL: entry m is row m) with a HOST count, and
 * entry m = t N + n selects the feature bytes of row n of step t and d_counters[t], as for wab_policy_backward (the noise
 * key is the global env id env_id_base + n). Their arrays are indexed by the list position m, so a minibatch needs no
 * [T, N] arrays; an entry may repeat (it then counts once per occurrence, so M may exceed T N). An entry outside
 * [0, T N) gets NaN logits and value and contributes nothing to the gradient.
 * wab_policy_evaluate writes d_logits f32[M][A] (the action head's output before the softmax, bias included) and d_value
 * f32[M]. It recomputes the forward with wab_policy_forward's arithmetic: under the weights a rollout used, d_value equals
 * what wab_policy_forward returned for that row bit for bit, and log_softmax(d_logits) its log-probabilities to rounding.
 * wab_policy_backward_logits writes d_grad f32 (layout as wab_policy_backward's) = the gradient of
 *   sum over m of  sum_o d_g_logits[m][o] logit_o(x_m) + d_g_value[m] V(x_m),
 * the same pass as wab_policy_backward with d heads taken as given. Its scratch is left as wab_policy_backward's, so
 * wab_policy_backward_grad_f64 (and wab_policy_grad_sum_ranks over ranks) apply to it. Neither call synchronises.
 * Arguments otherwise as for wab_policy_backward (wab_policy_evaluate takes no transposed weights; it needs the scratch
 * of wab_policy_backward_scratch_bytes for the hidden activations of its tiles). Equal inputs give bit-identical outputs.
 * WAB_E_NULL for a missing pointer (d_rows may be NULL); WAB_E_CONFIG for misalignment, too small a scratch,
 * n_rows < 0 or a negative or non-finite noise_scale; WAB_E_UNSUPPORTED beyond 8 actions, for hidden2 != 150 or
 * flat_dim > 512. */
int wab_policy_evaluate(WabVec *h, const uint8_t *d_features, int64_t n_steps, int64_t n_envs, const uint64_t *d_counters,
                        const int32_t *d_rows, int64_t n_rows, const void *d_packed1, const float *d_bias1,
                        const void *d_packed2, const float *d_bias2, int32_t hidden2, const void *d_packed3,
                        const float *d_bias3, const float *d_w_heads, const float *d_b_heads, int32_t n_actions,
                        float noise_scale, float leaky_slope, float clamp_lo, float clamp_hi, void *d_scratch,
                        int64_t scratch_bytes, float *d_logits, float *d_value, void *stream);
int wab_policy_backward_logits(WabVec *h, const uint8_t *d_features, int64_t n_steps, int64_t n_envs,
                               const uint64_t *d_counters, const int32_t *d_rows, int64_t n_rows, const float *d_g_logits,
                               const float *d_g_value, const void *d_packed1, const float *d_bias1, const void *d_packed2,
                               const float *d_bias2, int32_t hidden2, const void *d_packed3, const float *d_bias3,
                               const void *d_packed2t, const void *d_packed3t, const float *d_w_heads,
                               const float *d_b_heads, int32_t n_actions, float noise_scale, float leaky_slope,
                               float clamp_lo, float clamp_hi, void *d_scratch, int64_t scratch_bytes, float *d_grad,
                               void *stream);

/* Data-parallel training: the cross-rank gradient sum, deterministic and rounded once.
 * wab_policy_backward_grad_f64 reduces the scratch left by the last wab_policy_backward / wab_policy_ppo_backward /
 * wab_policy_backward_logits with this d_scratch on this stream into d_grad64 f64[n_params] (same layout as d_grad, the
 * same CTA order, the fp64 sums not rounded). wab_policy_grad_sum_ranks writes d_grad f32[n] = fp32(sum over r in index order of d_rank_grads[r][i]), the
 * sum in fp64, for an all-gathered d_rank_grads f64[n_ranks][n]. With one rank, sum_ranks(grad_f64) equals
 * wab_policy_backward's d_grad bit for bit. WAB_E_NULL for a missing pointer; WAB_E_CONFIG for misalignment (16 bytes
 * for d_scratch, 8 for the fp64 arrays, 4 for d_grad), too small a scratch, n_ranks < 1 or n < 0; WAB_E_UNSUPPORTED
 * beyond 8 actions or flat_dim > 512. */
int wab_policy_backward_grad_f64(WabVec *h, const void *d_scratch, int64_t scratch_bytes, int32_t n_actions,
                                 double *d_grad64, void *stream);
int wab_policy_grad_sum_ranks(const double *d_rank_grads, int32_t n_ranks, int64_t n, float *d_grad, void *stream);
/* wab_policy_backward_grad_f64 for a population: reduces the scratch left by the last wab_policy_ppo_backward_population of
 * n_members members with this d_scratch on this stream into d_grad64 f64[n_members][stride], stride =
 * wab_policy_population_grad_stride(h, n_actions), in the same element order as that call's d_grad, the fp64 sums not
 * rounded; the padding entries of every row are written as 0. With one rank, wab_policy_grad_sum_ranks over n =
 * n_members stride elements equals wab_policy_ppo_backward_population's d_grad bit for bit on every parameter.
 * WAB_E_NULL for a missing pointer; WAB_E_CONFIG for n_members outside [1, 64], misalignment (16 bytes for d_scratch, 8
 * for d_grad64) or a scratch smaller than wab_policy_backward_population_scratch_bytes(h, n_members); WAB_E_UNSUPPORTED
 * beyond 8 actions or flat_dim > 512. */
int wab_policy_backward_population_grad_f64(WabVec *h, const void *d_scratch, int64_t scratch_bytes, int32_t n_members,
                                            int32_t n_actions, double *d_grad64, void *stream);

/* The tail of the reference's Policy.forward + select_action (actor_critic.py:84-97, :108-125) for n_rows rows in one
 * pass, fp32: d_z3 f32[n_rows][128] is the PRE-activation output of affine3; x = clamp(leaky_relu(z3), lo, hi);
 * logits = W[0..A) x + b, value = W[A] x + b[A] (d_w_heads f32[A + 1][128] = action_head.weight stacked on
 * value_head.weight, d_b_heads f32[A + 1]); probs = softmax(logits); one action per row by inverse CDF on a uniform
 * keyed by (seed, row, *d_counter), row the LOCAL row (no handle, no shard). Outputs: d_actions u8[n_rows]; d_value f32[n_rows], d_probs f32[n_rows][A],
 * d_logp f32[n_rows] (log-probability of the sampled action) — each may be NULL. */
int wab_policy_tail(const float *d_z3, int32_t hidden, const float *d_w_heads, const float *d_b_heads, int64_t n_rows,
                    int32_t n_actions, float leaky_slope, float clamp_lo, float clamp_hi, uint64_t seed,
                    const uint64_t *d_counter, uint8_t *d_actions, float *d_value, float *d_probs, float *d_logp,
                    void *stream);

/* ---- Environment 2.0 ("/root/reference/Environment 2.0"): a toroidal W x H world of ostriches, wolves and
 * bushes per environment. One call = one world turn: every entity, in id order (ostriches, wolves, bushes),
 * observes and acts exactly as the reference driver loop does (Env2Tests.py:46-88: get_obs(i), take_action(i)). */
typedef struct Wab2Config {
    int32_t abi_version;
    int32_t width, height;                       /* World(width, height), World.py:141                              */
    int32_t n_ostriches, n_wolves, n_bushes;     /* create_ostriches / wolves / bushes, WAB_Environment2.py:61-110  */
    int32_t lookout_view_radius, gatherer_view_radius, wolf_view_radius;   /* WAB_Environment2.py:35-36, :49       */
    int32_t window_radius;                       /* R of the (2R+1)^2 observation window (>= the largest radius)    */
    int32_t starting_role;                       /* :19                                                             */
    int32_t ostrich_starting_food;               /* :32 (integer-valued in the reference's arithmetic)              */
    int32_t wolf_starting_food, wolf_food_for_eating_ostrich;   /* :43-44                                           */
    int32_t food_per_bush, food_given_per_turn;  /* :28-29, Bush.take_food Bush.py:31-39                            */
} Wab2Config;
typedef struct Wab2World Wab2World;
/* World.__init__ + create_* for n_envs worlds (keyed spawn positions). Synchronises. */
int wab2_create(const Wab2Config *cfg, int64_t n_envs, uint64_t seed, uint64_t env_id_base, int32_t device, Wab2World **out);
/* reset_environment (WAB_Environment2.py:113-118) of every world. */
int wab2_reset(Wab2World *h, void *stream);
/* One world turn. d_actions u8[A][N] is ENTITY-MAJOR, A = n_ostriches + n_wolves (bushes act with 0). Outputs per
 * acting entity, in the handle's output layout (wab2_output_layout): 0 = entity-major, d_planes u8[A][N][3][2R+1][2R+1]
 * (ostriches, wolves, bushes listed by get_observations at [dx+R][dy+R]; may be NULL), d_internal i32[A][N][5]
 * (x, y, food, role | is_running, status; may be NULL), d_reward f32[A][N], d_done u8[A][N] — the worlds of a warp
 * are contiguous; 1 = world-major, the same arrays with the first two dimensions exchanged ([N][A]...) — the A
 * windows of a world are one contiguous run for the warp that owns it. The observation of entity i is taken right
 * before it acts. */
int wab2_turn(Wab2World *h, const uint8_t *d_actions, uint8_t *d_planes, int32_t *d_internal, float *d_reward,
              uint8_t *d_done, void *stream);
/* Hidden state (tests, checkpoints): out9 i32[N][E][9] = type, x, y, table X, table Y, Visible, food, role, status;
 * turn and episode i32[N] (either may be NULL). Synchronises. */
int wab2_export_state(Wab2World *h, int32_t *out9, int32_t *turn, int32_t *episode, void *stream);
/* The inverse of wab2_export_state (tests: the reference's own known-answer worlds, World_tests.py:5-88, are built
 * from explicit positions; checkpoints): in9 i32[N][E][9] in the export layout (the type column must match the
 * handle's entity order: ostriches, wolves, bushes); turn, episode i32[N] or NULL (unchanged). Synchronises. */
int wab2_import_state(Wab2World *h, const int32_t *in9, const int32_t *turn, const int32_t *episode, void *stream);
/* Which kernel serves this handle: 0 = wab2_turn_kernel (one thread per world), 1 = wab2_grid_turn_kernel (one
 * warp per world with occupancy planes, for worlds every observation window fits once). Results are identical. */
int wab2_kernel_kind(const Wab2World *h);
/* Layout of wab2_turn's outputs for this handle: 0 = entity-major [A][N]..., 1 = world-major [N][A]... (the
 * warp-per-world kernel). */
int wab2_output_layout(const Wab2World *h);
void wab2_destroy(Wab2World *h);

/* Raw Philox4x32-10 on the device for n counters (cross-checks the RNG contract). d_ctr u32[n][4],
 * d_out u32[n][4]. */
int wab_philox_device(const uint32_t *d_ctr, uint32_t key0, uint32_t key1, int64_t n, uint32_t *d_out,
                      void *stream);

const char *wab_last_error(void);
int wab_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif
