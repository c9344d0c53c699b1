/*
 * ctf_b200.h — C ABI of the B200-native batched GridworldCtf step path.
 *
 * The reference (g-nightingale/marl-ctf-development) has no FFI layer: its
 * boundary is the duck-typed Python surface of `GridworldCtf`
 * (gridworld_ctf.py:19-52 ctor, :383 reset, :849-918 step, :975-1009
 * standardise_state, :1027-1069 get_env_metadata).  Each entry point below
 * names the reference member(s) it replaces.  The Python host
 * (marl_ctf_development_b200/env.py) binds these with ctypes; nothing in the
 * signatures is a torch type — plain pointers, sizes and a CUDA stream handle
 * passed as void*.
 *
 * Ownership: the caller owns every state and output buffer (device memory,
 * e.g. torch CUDA tensors).  The library owns only the opaque handle.
 * Threading: all calls are asynchronous on the given stream, never
 * synchronise the host (except the *_host entry points, which return when the
 * host buffers are valid) and never fall back to the CPU.
 * Errors: 0 = ok, negative = error; ctf_last_error() returns the message of
 * the last failing call on this thread.
 */
#ifndef CTF_B200_H
#define CTF_B200_H

#include <stddef.h>
#include <stdint.h>
#include <sys/types.h> /* ssize_t */

#ifdef __cplusplus
extern "C" {
#endif

#define CTF_ABI_VERSION 13

#define CTF_MAX_AGENTS 8    /* largest AGENT_STARTING_POSITIONS in scenarios.py has 8 entries */
#define CTF_MAX_GRID 16     /* GRID_SIZE <= 16 (shipped maps: 11, 13, 15) */
#define CTF_MAX_CELLS 256
#define CTF_N_TILE_CODES 14 /* gridworld_ctf.py:250-270: 0 open .. 13 team-1 flag */
#define CTF_MAX_CHANNELS 14 /* 1 self plane + at most 13 tile planes */
#define CTF_N_ACTIONS 9     /* gridworld_ctf.py:100-145 */
#define CTF_N_TYPES 4       /* 0 scout, 1 guardian, 2 vaulter, 3 miner (by behaviour) */
#define CTF_N_METRICS 13    /* agent-level counter families, gridworld_ctf.py:456-468 */

/* order of the per-agent counters in the stats buffer ([B][CTF_N_METRICS][N] u32) */
enum ctf_metric {
    CTF_M_TAG_COUNT = 0,
    CTF_M_RESPAWN_TAG_COUNT = 1,
    CTF_M_FLAG_PICKUPS = 2,
    CTF_M_FLAG_CAPTURES = 3,
    CTF_M_FLAG_DISPOSSESSIONS = 4,
    CTF_M_BLOCKS_LAID = 5,
    CTF_M_BLOCKS_MINED = 6,
    CTF_M_BLOCKS_LAID_DIST_OWN_FLAG = 7,
    CTF_M_BLOCKS_LAID_DIST_OPP_FLAG = 8,
    CTF_M_STEPS_DEFENDING_ZONE = 9,
    CTF_M_STEPS_ATTACKING_ZONE = 10,
    CTF_M_STEPS_ADJ_TEAMMATE = 11,
    CTF_M_STEPS_ADJ_OPPONENT = 12
};

/* bits of the device fault word (ctf_take_faults) */
#define CTF_FAULT_BAD_ACTION 1u      /* an action > 8 was passed (KeyError in ACTION_DELTAS, gridworld_ctf.py:710) */
#define CTF_FAULT_RESPAWN_BLOCKED 2u /* a lethal tag found no open cell in the victim's 3x3 spawn window: the
                                        reference raises ValueError from np.random.randint(0) (gridworld_ctf.py:771);
                                        here the victim stays where it is with HP <= 0 and the bit is set */
#define CTF_FAULT_BAD_INDEX 4u       /* a row of ctf_sample_actions named a flat_index outside [0, B*N); the row
                                        wrote nothing */

enum ctf_error {
    CTF_OK = 0,
    CTF_ERR_INVALID = -1, /* bad argument / config */
    CTF_ERR_CUDA = -2,    /* a CUDA runtime call failed */
    CTF_ERR_NO_DEVICE = -3
};

/* element type of the observation buffer; the values are {0, 1}, exact in every type */
enum ctf_obs_dtype { CTF_OBS_F32 = 0, CTF_OBS_U8 = 1, CTF_OBS_F16 = 2, CTF_OBS_BF16 = 3 };

/*
 * Compiled environment description: everything GridworldCtf.__init__ +
 * load_scenario + reset derive from (AGENT_CONFIG, SCENARIO, kwargs), flattened
 * to a POD.  Built on the host by marl_ctf_development_b200/config.py.
 * HP quantities are fixed point: value_q = value * hp_scale (exact for every
 * shipped config; the compiler refuses configs where it is not).
 */
typedef struct ctf_config {
    /* 8-byte members first so that C, CUDA and ctypes agree on the layout */
    uint64_t tag_threshold;     /* #32-bit words w with w/2^32 < TAG_PROBABILITY  (:815) */
    double reward_step;         /* REWARD_STEP (:78) */
    double reward_capture;      /* REWARD_CAPTURE (:77) */
    double reward_tag;          /* REWARD_TAG (:79) */
    double capture_punish;      /* 1.0 * REWARD_CAPTURE * OPP_FLAG_CAPTURE_PUNISHMENT_SCALAR (:964) */
    double win_margin_scalar;   /* WIN_MARGIN_SCALAR (:75) */
    double loss_margin_scalar;  /* LOSS_MARGIN_SCALAR (:76) */

    int32_t grid_size;          /* G */
    int32_t n_agents;           /* N */
    int32_t n_channels;         /* C = 1 + len(TILES_USED)  (:1016) */
    int32_t game_steps;         /* GAME_STEPS */
    int32_t flip_axis;          /* FLIP_AXIS: -1 = None (both axes), 0 rows, 1 cols, 2 anti-diagonal (:1003-1007) */
    int32_t use_adjusted_rewards;
    int32_t home_flag_capture;
    int32_t drop_flag_when_no_hp;
    int32_t hp_scale;
    int32_t heal_q;             /* AGENT_HP_HEALING_PER_STEP */
    int32_t vault_cost_q;       /* VAULT_HP_COST */
    int32_t vault_min_q;        /* VAULT_MIN_HP */
    int32_t zone_distance;      /* DEFENSIVE_ZONE_DISTANCE (:87) */
    int32_t guardian_distance;  /* GUARDIAN_DEFENSE_DISTANCE (:226) */
    int32_t tagging_range;      /* GUARDIAN_TAGGING_RANGE (:227) */
    int32_t max_agent_blocks;   /* MAX_AGENT_BLOCKS (:241) */
    int32_t block_pickup_value; /* BLOCK_PICKUP_VALUE (:85) */
    int32_t reverse_team1_actions; /* 1: step() maps team-1 actions through reversed_action first (:968-973) */
    int32_t hp_max_q[CTF_N_TYPES];         /* AGENT_TYPE_HP */
    int32_t damage_q[CTF_N_TYPES];         /* AGENT_TYPE_DAMAGE */
    int32_t damage_boosted_q[CTF_N_TYPES]; /* AGENT_TYPE_DAMAGE * GUARDIAN_DAMAGE_MULTIPLIER */

    uint8_t agent_team[CTF_MAX_AGENTS];
    uint8_t agent_type[CTF_MAX_AGENTS];
    uint8_t agent_tile[CTF_MAX_AGENTS];    /* AGENT_TILE_MAP (:264) */
    uint8_t start_row[CTF_MAX_AGENTS];
    uint8_t start_col[CTF_MAX_AGENTS];
    uint8_t obs_reverse[CTF_MAX_AGENTS];   /* reverse_grid flag used for agent i's observation (callers: team != 0) */
    uint8_t meta_hp_src[CTF_MAX_AGENTS];   /* agent id whose HP feeds metadata slot i: = type of agent i (:1040-1041 quirk) */
    uint8_t n_opponents[2];                /* len(OPPONENTS[t]) (:391-395) */
    uint8_t opponents[2][CTF_MAX_AGENTS];  /* OPPONENTS[t] in id order */
    uint8_t flag_pos[2][2];                /* FLAG_POSITIONS */
    uint8_t capture_pos[2][2];             /* CAPTURE_POSITIONS */
    uint8_t spawn_pos[2][2];               /* SPAWN_POSITIONS */
    uint8_t flag_tile[2];                  /* FLAG_TILE_MAP: 12, 13 */
    int8_t action_delta[CTF_N_TYPES][CTF_N_ACTIONS][2]; /* ACTION_DELTAS (:100-145) */
    uint8_t reversed_action[CTF_N_ACTIONS + 7];          /* REVERSED_ACTION_MAP[FLIP_AXIS], padded to 16 */
    uint8_t type_action_mask[CTF_N_TYPES];               /* AGENT_TYPE_ACTION_MASK (:218-223) */
    uint8_t chan_lut[2][16];               /* [observer team][tile code] -> channel 1..C-1, 0 = no channel (O1) */
    uint8_t grid_template[CTF_MAX_CELLS];  /* load_scenario() result, row-major G x G */

    /* HP representation.  0: exact fixed point (the *_q fields, hp_scale) — every shipped configuration.  1: IEEE doubles
       (the *_f fields below), for HP / damage / heal / vault quantities that are not dyadic rationals (e.g. heal 0.1):
       the device then performs the reference's Python float operations one by one (gridworld_ctf.py:648-657, 818-824,
       785, 845-846, 1040) and keeps HP in state.hp. */
    int32_t hp_float;
    int32_t reserved0;
    double hp_max_f[CTF_N_TYPES];          /* AGENT_TYPE_HP */
    double damage_f[CTF_N_TYPES];          /* AGENT_TYPE_DAMAGE */
    double damage_boosted_f[CTF_N_TYPES];  /* AGENT_TYPE_DAMAGE * GUARDIAN_DAMAGE_MULTIPLIER (one float multiplication) */
    double heal_f, vault_cost_f, vault_min_f;
} ctf_config_t;

/* Device buffers of the B resident environments (SoA of field groups, env-major). */
typedef struct ctf_state {
    uint8_t* grid;    /* [B][grid_stride] tile codes, grid_stride = ctf_sizes.grid_stride */
    uint64_t* agents; /* [B][N] packed: row | col<<8 | has_flag<<16 | hp_q(int16)<<32 | inventory(uint16)<<48 */
    uint32_t* envs;   /* [B][4]: env_step_count, episode, team_flag_captures[0], team_flag_captures[1] */
    uint32_t* stats;  /* [B][13][N] counters, or NULL when created with stats_level 0 */
    uint8_t* visits;  /* [B][N][G*G] uint8 visitation maps (wrap at 256), or NULL unless stats_level 2 */
    double* hp;       /* [B][N] agent HP as doubles when cfg.hp_float is set (the hp_q field of `agents` is then unused), else NULL */
} ctf_state_t;

/* Device output buffers of one reset()/step(). Any pointer may be NULL to skip that output. */
typedef struct ctf_outputs {
    void* obs;        /* [B][N][C][G][G] float32 (or uint8 / float16 / bfloat16): standardise_state(i, obs_reverse[i]) for every agent */
    uint32_t* obs_bits; /* [B][N][bits_words_per_agent] packed copy of the same observations, 1 bit per element:
                         element c*G*G + p of agent a is bit (c*G*G + p) % 32 of word a*wpa + (c*G*G + p) / 32.
                         For rollout storage (32x smaller than float32); ctf_unpack_obs expands it. */
    float* meta;      /* [B][N][6+2N] float32: get_env_metadata(i) (fp16-rounded values) */
    float* rewards;   /* [B][N] float32 */
    uint8_t* dones;   /* [B] 0/1 */
} ctf_outputs_t;

typedef struct ctf_sizes {
    size_t grid_stride;  /* bytes per env in state.grid (G*G padded to 16) */
    size_t grid_bytes, agents_bytes, envs_bytes, stats_bytes, visits_bytes;
    size_t obs_bytes, meta_bytes, rewards_bytes, dones_bytes;
    size_t obs_elems_per_env, meta_elems_per_env;
    size_t obs_bits_bytes;       /* bytes of outputs.obs_bits */
    size_t bits_words_per_agent; /* ceil(C*G*G / 32) */
    size_t hp_bytes;             /* bytes of state.hp (0 unless cfg.hp_float) */
} ctf_sizes_t;

typedef struct ctf_env* ctf_handle_t;

const char* ctf_last_error(void);
int ctf_abi_version(void);

/* Number of bytes of ctf_config_t this library was built with (layout check for bindings). */
size_t ctf_config_size(void);

/*
 * Replaces GridworldCtf.__init__ (gridworld_ctf.py:19-350) for a batch:
 * validates cfg, selects `device`, keeps (seed, env_id_base) as the counter-RNG
 * key/offset (env b draws with id env_id_base + b, so results do not depend on
 * how envs are sharded over GPUs).  stats_level: 0 none, 1 counters, 2 counters
 * + visitation maps.  obs_dtype: ctf_obs_dtype.
 */
int ctf_create(const ctf_config_t* cfg, int64_t num_envs, int device, uint64_t seed,
               uint64_t env_id_base, int stats_level, int obs_dtype, ctf_handle_t* out);
int ctf_destroy(ctf_handle_t h);

/* Buffer sizes the caller must allocate (replaces get_env_dims, gridworld_ctf.py:1011-1025). */
int ctf_get_sizes(ctf_handle_t h, ctf_sizes_t* out);

/*
 * Replaces GridworldCtf.reset (gridworld_ctf.py:383-477): every env back to the
 * scenario's initial state, episode counter + 1 (first reset -> episode 0 when
 * `first` is non-zero), statistics cleared; writes observations/metadata of
 * the initial state, zero rewards and dones.
 */
int ctf_reset(ctf_handle_t h, ctf_state_t state, ctf_outputs_t out, int first, void* stream);

/*
 * Replaces GridworldCtf.step (gridworld_ctf.py:849-918) followed by
 * standardise_state + get_env_metadata for every agent (ppo.py:66-95,
 * utils.py:528-551).  actions: device uint8 [B][N], values 0..8 (values > 8,
 * which raise KeyError in the reference, set bit 0 of the handle's fault word
 * and are treated as no-op 4).
 */
int ctf_step(ctf_handle_t h, ctf_state_t state, const uint8_t* actions, ctf_outputs_t out, void* stream);

/*
 * Replaces standardise_state(i, reverse_grid) / get_env_metadata(i) called on
 * their own: observations of the current state without stepping.
 * reverse_flags: host uint8 [N] (NULL = cfg.obs_reverse).
 */
int ctf_observe(ctf_handle_t h, ctf_state_t state, const uint8_t* reverse_flags, ctf_outputs_t out, void* stream);

/*
 * Expands packed observations (outputs.obs_bits layout, any number of agent blocks, e.g. a minibatch gathered
 * from a rollout buffer) into out[n_agent_blocks][C][G][G] of ctf_obs_dtype out_dtype — what the policy
 * consumes at PPO update time (ppo.py:298, 440) without ever holding the float32 rollout in memory.
 */
int ctf_unpack_obs(ctf_handle_t h, const uint32_t* packed, void* out, int out_dtype, int64_t n_agent_blocks, void* stream);

/*
 * Sum of the per-env counters over this handle's envs: device int64
 * [13][N] written to stats_sum (replaces the per-episode harvest of
 * env.metrics, metrics_logger.py:137-159); the caller all-reduces it over ranks.
 */
int ctf_stats_sum(ctf_handle_t h, ctf_state_t state, int64_t* stats_sum, void* stream);

/* Reads and clears the device fault word (CTF_FAULT_* bits). Synchronises the stream. */
int ctf_take_faults(ctf_handle_t h, void* stream, uint32_t* faults);

/*
 * Host-buffer variant of ctf_step for callers that keep actions and rewards on
 * the host: actions_host ([B][N] uint8) in, rewards ([B][N] float32) and dones
 * ([B] uint8) out, valid when the call returns.  Pinned (page-locked) buffers
 * are accessed by the kernel directly over PCIe; pageable ones are staged with
 * copies.  Observations and metadata stay on the device in `out`.
 * One handle must not have two steps in flight on different streams: the
 * host-step staging buffers are per handle.
 */
int ctf_step_host(ctf_handle_t h, ctf_state_t state, const uint8_t* actions_host, ctf_outputs_t out,
                  float* rewards_host, uint8_t* dones_host, void* stream);

/*
 * Observation record (ABI 13): lets ctf_step store only the 32-byte sectors of `obs` that changed since the last
 * write, which are about 1 % of them.  The caller keeps, for one observation buffer it owns:
 *   record        device [B][ctf_obs_record_size / (4 B)] uint32, 16-byte aligned: per env, the padded bit string
 *                 the last launch wrote into obs (contents need no initialisation);
 *   record_epoch  device [B] uint32: the epoch in which each env's record was written;
 *   epoch         device uint32: the current epoch.
 * An env's record is valid when record_epoch[env] == *epoch.  A launch whose outputs.obs equals the bound `obs`
 * (ctf_step, ctf_step_host, ctf_reset, ctf_observe) writes an env with a valid record as a delta (ctf_step and
 * ctf_step_host) and any other env in full (all four), then refreshes the record and stamps record_epoch.  Every
 * launch into another buffer writes exactly as without a record.  The contract: between two such launches nothing
 * else may write `obs` unless *epoch is changed first (in stream order, e.g. by adding 1 on the device, which a CUDA
 * graph can capture); otherwise the next delta leaves the foreign bytes in place.
 * obs = NULL unbinds (record, record_epoch, epoch are then ignored).  Rejected with CTF_ERR_INVALID: a null handle; a
 * non-null obs with a null record, record_epoch or epoch; record not 16-byte, record_epoch or epoch not 4-byte aligned;
 * any two of obs (the handle's dense size), record, record_epoch and epoch overlapping.  The handle keeps the pointers,
 * not the memory: unbind before freeing it.
 */
int ctf_bind_obs_record(ctf_handle_t h, const void* obs, uint32_t* record, uint32_t* record_epoch, const uint32_t* epoch);
/* Bytes of the record ctf_bind_obs_record needs for this handle: B * (padded bit-string words per env) * 4. */
int ctf_obs_record_size(ctf_handle_t h, size_t* record_bytes);

/*
 * Policy inference from packed observations (no reference counterpart: the reference feeds agent_network.Agent a dense
 * float32 grid).  Weights of the convolutional trunk of policy.CtfPolicy; all pointers are device memory, none null,
 * conv1_w 16-byte, conv2_w 8-byte and the biases 4-byte aligned.
 */
typedef struct ctf_policy_weights {
    const float* conv1_w;   /* [16][C][3][3] fp32 (conv1.weight as stored by torch) */
    const float* conv1_b;   /* [16] */
    const void*  conv2_w;   /* bf16 [9 taps][4 n-tiles][32 lanes][4], the mma.sync B-fragment order that
                               fused_policy.conv2_kernel_layout_index() gives from conv2.weight [32][16][3][3] */
    const float* conv2_b;   /* [32] */
} ctf_policy_weights_t;

/*
 * Trunk of CtfPolicy (conv1 -> tanh -> conv2 -> tanh -> flatten, then the metadata) computed from packed
 * observations: writes one bf16 feature row per sample, [32*(G-4)^2 conv2 outputs in (c, y, x) order | M metadata
 * values | zeros up to feature_stride], i.e. the fc1 input.  Sample s = e*k + j (e < n_envs, j < k) reads packed
 * block e*agents_per_env + agent_ids[j] ([bits_words_per_agent] uint32, outputs.obs_bits layout) and the metadata row
 * ([M] float32) with the same index: agents_per_env = N with a team's ids reads outputs.obs_bits / outputs.meta in
 * place, agents_per_env = 1 with id 0 reads contiguous rows (e.g. a rollout buffer).
 * conv1 is exact fp32 sparse accumulation over the set bits (any {0,1} input), tanhf, rounded to bf16; conv2 runs on
 * tensor cores (bf16 inputs and weights, fp32 accumulation, fp32 bias, tanhf, rounded to bf16).  Deterministic (no
 * atomics), no allocation and no host synchronisation: capturable in a CUDA graph.
 * agent_ids: host array of k (1..8) ids < agents_per_env.  features: 16-byte aligned; feature_stride: elements per
 * row, a multiple of 8 and >= 32*(G-4)^2 + M.
 */
int ctf_policy_features(ctf_handle_t h, const ctf_policy_weights_t* w, const uint32_t* packed, const float* meta,
                        int64_t n_envs, int agents_per_env, const uint8_t* agent_ids, int k,
                        void* features, int64_t feature_stride, void* stream);

/*
 * Grouped trunk: ctf_policy_features for many segments, each with its own policy, in one launch (league evaluation
 * and every other workload that runs several policies on one env batch).  A segment names a policy (an index into
 * the weights table), an env range, k agent ids and the feature row of its sample 0.  Its sample s = e*k + j
 * (e < n_envs, j < k) reads packed block (env_begin + e)*agents_per_env + agent_ids[j] and the metadata row with the
 * same index, as ctf_policy_features does, and writes feature row out_row + s.  Every row is bit-identical to what
 * ctf_policy_features writes with that segment's weights for the same sample (both entry points run the same kernel).
 * Rows outside every segment are not written.
 * Scheduling: the samples are cut into tiles of 8 consecutive samples of one segment, in table order; every CTA takes
 * a contiguous range of tiles and restages conv weights in shared memory only where the policy changes, so put the
 * segments of one policy next to each other.  Deterministic (no atomics), no allocation and no host synchronisation:
 * capturable in a CUDA graph; the tables are validated on the host and passed by value as kernel parameters, so a
 * captured graph keeps its own copy.
 * Limits: 1..CTF_GROUPED_MAX_POLICIES policies and 1..CTF_GROUPED_MAX_SEGMENTS segments per call (the tables fill
 * about 26 KB of the 32 764 bytes of kernel parameters).
 * Rejected with CTF_ERR_INVALID: a policy index out of range; k outside 1..8 or an id >= agents_per_env; an env range
 * outside [0, n_envs); output rows outside [0, n_rows) or two segments whose rows overlap; feature_stride or features
 * as ctf_policy_features requires them; null or misaligned weights or inputs; too many policies or segments.
 * Segments with n_envs = 0 are allowed; when every segment is empty nothing is launched.
 */
#define CTF_GROUPED_MAX_POLICIES 64
#define CTF_GROUPED_MAX_SEGMENTS 512

typedef struct ctf_policy_segment {
    int64_t env_begin;   /* first env of the segment */
    int64_t n_envs;      /* envs of the segment (>= 0) */
    int64_t out_row;     /* feature row of the segment's sample 0 */
    int32_t policy;      /* index into the weights table */
    int32_t k;           /* 1..8 agents per env */
    uint8_t agent_ids[CTF_MAX_AGENTS];   /* the first k are read */
} ctf_policy_segment_t;

/* weights: host table of n_policies ctf_policy_weights_t (device pointers); segments: host table of n_segments;
   n_envs: envs in the packed / meta buffers; n_rows: rows of the feature buffer. */
int ctf_policy_features_grouped(ctf_handle_t h, const ctf_policy_weights_t* weights, int n_policies,
                                const ctf_policy_segment_t* segments, int n_segments, const uint32_t* packed,
                                const float* meta, int64_t n_envs, int agents_per_env, void* features,
                                int64_t feature_stride, int64_t n_rows, void* stream);

/* CTAs the trunk kernel runs at most per launch on this handle (the device's SMs times the CTAs resident per SM for
   this plan, counted at ctf_create), for each of its two instantiations: trunk_ctas for launches with one policy and
   one segment (every ctf_policy_features call), grouped_ctas for every other ctf_policy_features_grouped call. */
int ctf_policy_trunk_ctas(ctf_handle_t h, int* trunk_ctas, int* grouped_ctas);

/* fp32 gradients of the trunk's parameters in torch layout (device memory). */
typedef struct ctf_policy_grads {
    float* conv1_w;   /* [16][C][3][3] */
    float* conv1_b;   /* [16] */
    float* conv2_w;   /* [32][16][3][3] */
    float* conv2_b;   /* [32] */
} ctf_policy_grads_t;

/* Bytes of device workspace ctf_policy_features_backward needs on this handle (fixed per handle: one row of partial
   sums per CTA of the backward kernel, a count taken from the device's occupancy at ctf_create). */
int ctf_policy_grad_workspace_size(ctf_handle_t h, size_t* bytes);

/*
 * Backward of ctf_policy_features for training: the gradients of conv1 / conv2 weights and biases given the
 * gradient of the loss with respect to the feature rows.  Same sample -> block addressing as ctf_policy_features.
 * features: the rows ctf_policy_features wrote for these samples with the weights `w` (their conv2 outputs are h2);
 * grad_features: bf16 [n_samples][feature_stride], only columns < 32*(G-4)^2 are read (metadata and pad columns have no
 * parameters).  conv2_w_t: bf16 [9 taps][2 k-halves][2 n-tiles][32 lanes][4], conv2.weight in the transposed
 * mma.sync B-fragment order of fused_policy.conv2_transpose_layout_index().
 * Per sample: h1 = bf16(tanh(conv1)) recomputed bit for bit as the forward computes it; dz2 = bf16(dF * (1 - h2^2))
 * (fp32 operations); dW2 and db2 accumulate dz2 (x) h1 in fp32 on tensor cores; dh1 = conv2^T(dz2) on tensor cores
 * (bf16 weights, fp32 accumulation); dz1 = dh1 * (1 - h1^2) in fp32; dW1 and db1 are exact fp32 sums of dz1 over the
 * set input bits.  Per-CTA partial sums go to `workspace` (>= ctf_policy_grad_workspace_size bytes, 16-byte aligned)
 * and are summed in a fixed order: reruns are bit-identical (no atomics).  The gradient buffers are overwritten, not
 * accumulated into; n_envs = 0 writes zeros.  No allocation and no host synchronisation.
 */
int ctf_policy_features_backward(ctf_handle_t h, const ctf_policy_weights_t* w, const void* conv2_w_t,
                                 const uint32_t* packed, int64_t n_envs, int agents_per_env, const uint8_t* agent_ids,
                                 int k, const void* features, const void* grad_features, int64_t feature_stride,
                                 void* workspace, size_t workspace_bytes, const ctf_policy_grads_t* grads, void* stream);

/*
 * Generalised advantage estimation (GAE) over a rollout, on the device.  Layout of a collect_rollout buffer:
 * rewards, values, advantages and returns are fp32 [n_steps * agents_per_step][n_envs], row t*agents_per_step + j =
 * trained agent j at step t; next_value is fp32 [agents_per_step][n_envs], the bootstrap V(s_T) of every (agent, env)
 * (0 when the rollout ended the episode).  Each (agent, env) column is its own sequence over t; there is no done
 * input, for rollouts whose envs end only together at their last step (ctf_gae_dones takes one).  Backwards over t,
 * with nv = next_value at t = n_steps - 1 and values[t + 1] below it:
 *     delta = (rewards[t] + gamma*nv) - values[t];  last = delta + gamma_lambda*last (last = 0 before the first row);
 *     advantages[t] = last;  returns[t] = last + values[t]
 * Every operation is rounded on its own (no fused multiply-add), so the result is bit for bit what eager torch computes
 * for the same statements on fp32 tensors with Python scalars gamma and gamma*lambda: pass gamma = (float)gamma and
 * gamma_lambda = (float)(gamma * lambda computed in double).
 * Rejected with CTF_ERR_INVALID: a null pointer; n_steps < 1; agents_per_step outside 1..CTF_MAX_AGENTS; n_envs < 1;
 * gamma or gamma_lambda not finite or outside [0, 1]; a buffer not 4-byte aligned; an output that overlaps an input
 * or the other output.  No allocation and no host synchronisation (can be captured in a CUDA graph).
 */
int ctf_gae(ctf_handle_t h, const float* rewards, const float* values, const float* next_value, float* advantages,
            float* returns, int64_t n_steps, int64_t agents_per_step, int64_t n_envs, float gamma, float gamma_lambda,
            void* stream);

/*
 * ctf_gae for rollouts that cross episode boundaries (ABI 11).  dones is fp32 [n_steps * agents_per_step][n_envs],
 * the layout of rewards; a nonzero dones[t*agents_per_step + j][b] means that observation t of (agent j, env b)
 * starts a new episode (CleanRL's convention).  The recurrence is ctf_gae's, except that after row t, when dones[t]
 * is nonzero, nv and last both become exactly 0 (a select, not a multiply by 1 - dones) before row t - 1:
 *     delta = (rewards[t] + gamma*nv) - values[t];  last = delta + gamma_lambda*last;
 *     advantages[t] = last;  returns[t] = last + values[t];  nv = values[t];
 *     if (dones[t] != 0) nv = last = 0
 * next_value is the bootstrap of the last row, so pass 0 where the last step ended the episode.  dones[0] changes
 * nothing in this rollout.  With all dones zero the result is bit for bit ctf_gae's, which reads 4 fewer bytes per
 * element.  Rejected as ctf_gae rejects, and also: a null dones, a dones not 4-byte aligned, an output that overlaps
 * dones.  No allocation and no host synchronisation.
 */
int ctf_gae_dones(ctf_handle_t h, const float* rewards, const float* values, const float* dones, const float* next_value,
                  float* advantages, float* returns, int64_t n_steps, int64_t agents_per_step, int64_t n_envs,
                  float gamma, float gamma_lambda, void* stream);

/*
 * Seeded action sampling for policy rows (ABI 12): one categorical draw per row from the value | logits head output,
 * with counter-based randomness like the env's, so that a rollout or duel is a function of its seeds alone.
 * head: fp32 [n_rows][head_stride], column 0 the value (not read), columns 1..9 the logits.  masked: uint8 [n_rows] or
 * NULL; a nonzero flag applies CtfPolicy.masked_logits (x_i += -1e9f for i >= 5, one fp32 add).  flat_index: int64
 * [n_rows], env * N + agent of every row (env b = flat_index / N, agent a = flat_index % N, env b of this handle).
 * Per row, with x the (masked) logits:
 *   u = (w0 >> 8) * 2^-24, w0 = word 0 of Philox4x32-10 with key (seed & 0xffffffff, seed >> 32) and counter
 *       (env_id_base + b, episode[b], env_step_count[b], 0x80000000 | a), the counts read from state.envs on the device
 *       at launch (a captured CUDA graph draws fresh words at every replay; the site's top bit keeps these counters apart
 *       from the env's sites 0..31 even when seed is the env's seed);
 *   m = max x;  e_i = expf(x_i - m);  c_i = e_0 + ... + e_i in fp32, ascending;  Z = c_8;
 *   action = the smallest i with u*Z < c_i; if none (rounding), the largest i with e_i > 0; if none (NaN or infinite
 *            logits), the no-op 4.  So the action is always in 0..8, and a masked row with finite logits takes 0..4;
 *   logprob = (x_action - m) - logf(Z);  entropy = logf(Z) - (sum over e_i > 0 of e_i * (x_i - m)) / Z.
 * Every add and multiply is rounded on its own (no FMA).  Outputs, each optional (NULL skips it): actions uint8
 * [B][N], written at flat_index; action_out int64, logprob and entropy fp32, [n_rows] each.  A row's outputs depend only
 * on its logits, its mask flag and (seed, global env id, episode, step, agent): not on n_rows, the row order or the
 * other rows, and reruns are bit-identical.  No allocation and no host synchronisation (capturable in a CUDA graph).
 * A flat_index outside [0, B*N) is a device-side error: that row writes nothing and sets CTF_FAULT_BAD_INDEX.
 * Rejected with CTF_ERR_INVALID: a null handle, state.envs, head or flat_index; n_rows < 0; head_stride < 10;
 * state.envs not 16-byte, flat_index or action_out not 8-byte, head, logprob or entropy not 4-byte aligned; an output
 * that overlaps an input (head, masked, flat_index) or another output.  n_rows = 0 launches nothing.
 */
int ctf_sample_actions(ctf_handle_t h, ctf_state_t state, const float* head, int64_t head_stride, const uint8_t* masked,
                       const int64_t* flat_index, int64_t n_rows, uint64_t seed, uint8_t* actions, int64_t* action_out,
                       float* logprob, float* entropy, void* stream);

/*
 * Compressible device memory for the dense observation buffer.  On devices with Compute Data Compression the memory
 * is compressed between L2 and DRAM, invisibly to every kernel and reader: the bytes read back are the bytes written.
 * The observations are mostly zero sectors, so their store stream moves far fewer DRAM bytes (DESIGN §4).
 * The two allocation entry points have the signatures torch.cuda.memory.CUDAPluggableAllocator expects (the stream
 * is unused).  ctf_compressible_alloc maps `size` bytes, rounded up to the allocation granularity, with
 * cuMemCreate / cuMemAddressReserve / cuMemMap / cuMemSetAccess (read-write for `device`).  It asks for
 * CU_MEM_ALLOCATION_COMP_GENERIC when the device reports support and compression is enabled, and otherwise, or when
 * the driver does not grant it, maps ordinary memory on the same path, so ctf_compressible_free releases either kind.
 * Returns NULL on failure (ctf_last_error has the reason).  The driver entry points are resolved through the CUDA
 * runtime: the library does not link libcuda.
 */
void* ctf_compressible_alloc(ssize_t size, int device, void* stream);
/* Unmaps and releases a pointer ctf_compressible_alloc returned; `size` is the size it was asked for. */
void ctf_compressible_free(void* p, ssize_t size, int device, void* stream);
/* *out = 1 when `device` reports CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, else 0. */
int ctf_compression_supported(int device, int* out);
/* *out = 1 when `p` lies in a cuMemMap'ed allocation whose properties say CU_MEM_ALLOCATION_COMP_GENERIC, else 0
   (also for memory from cudaMalloc or the host). */
int ctf_mem_is_compressed(const void* p, int* out);
/* enabled = 0 makes later ctf_compressible_alloc calls map ordinary memory, the path of devices without compression
   (tests of that path and A/B measurements); 1 (the default) restores compression.  Returns the previous setting. */
int ctf_compressible_set_enabled(int enabled);

#ifdef __cplusplus
}
#endif
#endif /* CTF_B200_H */
