/*
 * ngw.h — C-ABI of the B200-native batched NovelGridworld simulator (libngw_b200.so)
 *
 * One header, three users:
 *   - gym_novel_gridworlds_b200/csrc/ *.cu*  the sm_100a kernels and the C-ABI library (the product),
 *   - oracle/ngw_oracle.c                    the CPU restatement used ONLY as the parity checker,
 *   - gym_novel_gridworlds_b200/capi.py      ctypes mirror of these structs (the Python host layer).
 *
 * The reference (gtatiya/gym-novel-gridworlds, pure Python) has no FFI layer; its boundary for this
 * path is the gym-0.18 Python API.  The entry points below are what a maintainer of the reference
 * would bind (ctypes stub in INTEGRATION.md) to replace:
 *
 *   ngw_create / ngw_destroy      <- gym.make + wrapper constructors            (__init__.py:7-60,
 *                                     pogostick_v1_env.py:26-84, bow_v1_env.py:26-82,
 *                                     wrappers.py:63-68, observation_wrappers.py:16-30,
 *                                     novelty_wrappers.py:1586-1674)
 *   ngw_reset                     <- Env.reset + novelty reset overrides       (pogostick_v1_env.py:86-181,
 *                                     novelty_wrappers.py:29,456,664,868,904,1013,1071,1126,1161)
 *   ngw_step / ngw_step_host      <- Env.step through the whole wrapper chain  (pogostick_v1_env.py:230-367,
 *                                     bow_v1_env.py:228-340, wrappers.py:74-85,
 *                                     observation_wrappers.py:32-80, novelty_wrappers.py step methods)
 *   ngw_observe                   <- LidarInFront.observation                  (observation_wrappers.py:70-80)
 *   ngw_load_state / ngw_export_state / ngw_state
 *                                 <- the `env=` restore branch of reset / get_observation's live
 *                                     references                              (pogostick_v1_env.py:89-109,214-228)
 *   ngw_stats                     <- (absent in the reference; episode statistics for the NCCL reduce)
 *
 * All wrapper / novelty semantics are flattened by the host layer into one `ngw_config` per distinct
 * wrapper chain ("config"); every env of a batch carries a config id, so mixed-novelty batches run in
 * one launch.  No torch types appear here: plain pointers, sizes and a cudaStream_t passed as void*.
 */
#ifndef NGW_H
#define NGW_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NGW_ABI_VERSION 13

#define NGW_MAX_ITEMS 24          /* reference asserts len(items) <= 20 (pogostick_v1_env.py:75,220) */
#define NGW_MAX_ACTIONS 48
#define NGW_MAX_RECIPES 8
#define NGW_MAX_RECIPE_INPUTS 4
#define NGW_MAX_LAYERS 4
#define NGW_MAX_PLACE 12
#define NGW_MAX_RESET_OPS 8
#define NGW_MAX_MAP_SIZE 64
#define NGW_NONE 0xFF

/* ---- facing ids (pogostick_v1_env.py:33) ---- */
enum { NGW_NORTH = 0, NGW_SOUTH = 1, NGW_WEST = 2, NGW_EAST = 3 };

/* ---- terminal opcodes: what an external action id finally executes on the base env ---- */
enum ngw_op {
    NGW_OP_INVALID = 0,        /* id rejected by LimitActions (wrappers.py:76) or unknown to the base (pogostick_v1_env.py:236) */
    NGW_OP_NOOP = 1,           /* id known but no branch of the if/elif chain matches (pogostick_v1_env.py:244-347) */
    NGW_OP_FORWARD = 2,        /* pogostick_v1_env.py:244-257 */
    NGW_OP_LEFT = 3,           /* pogostick_v1_env.py:258-268 */
    NGW_OP_RIGHT = 4,          /* pogostick_v1_env.py:269-279 */
    NGW_OP_BREAK = 5,          /* pogostick_v1_env.py:280-294 and the novelty Break overrides (variant) */
    NGW_OP_PLACE_TREE_TAP = 6, /* pogostick_v1_env.py:295-314 */
    NGW_OP_EXTRACT_RUBBER = 7, /* pogostick_v1_env.py:315-331; arg = rubber gained (novelty_wrappers.py:1537-1551) */
    NGW_OP_EXTRACT_STRING = 8, /* bow_v1_env.py:293-304;      arg = string gained (novelty_wrappers.py:1524-1536) */
    NGW_OP_CRAFT = 9,          /* pogostick_v1_env.py:413-474 / novelty_wrappers.py:371-436; arg = recipe slot */
    NGW_OP_SELECT = 10,        /* pogostick_v1_env.py:338-347; arg = item id */
    NGW_OP_CHOP = 11,          /* novelty_wrappers.py:1288-1307 */
    NGW_OP_JUMP = 12           /* novelty_wrappers.py:1360-1382 */
};

/* ---- Break variants (which class's Break block is the outermost terminal interceptor) ---- */
enum ngw_break_variant {
    NGW_BRK_BASE = 0,          /* pogostick_v1_env.py:280-294: reward only for tree_log */
    NGW_BRK_AXE = 1,           /* novelty_wrappers.py:45-84 (AxeEasy/Medium/Hard), arg = axe item id */
    NGW_BRK_AXE_INC = 2,       /* same with breakincrease == 'true' */
    NGW_BRK_AXETOBREAK = 3,    /* novelty_wrappers.py:472-504, arg = axe item id */
    NGW_BRK_INCREASE = 4       /* novelty_wrappers.py:1434-1458, arg = itemtobreakmore id or NGW_NONE (= all) */
};

/* ---- pass-through layers wrapped around a terminal opcode, outermost first ---- */
enum ngw_layer {
    NGW_LAYER_END = 0,
    NGW_LAYER_CRATE = 1,       /* novelty_wrappers.py:1085-1088: pre-effect on Break when the front block is a crate */
    NGW_LAYER_FIREWALL = 2,    /* novelty_wrappers.py:1169-1189: post-check after the inner step */
    NGW_LAYER_FENCE_MEDIUM = 3,/* novelty_wrappers.py:918-973 with difficulty 'medium' */
    NGW_LAYER_FENCE_HARD = 4   /* novelty_wrappers.py:918-973 with difficulty 'hard' */
};

/* ---- reset post-processing ops, applied inner -> outer in wrap order ---- */
enum ngw_reset_kind {
    NGW_RESET_FENCE = 1,       /* novelty_wrappers.py:868-889: a = fence id, percent in [lo, hi) of non-air non-wall cells */
    NGW_RESET_ADDITEM = 2,     /* novelty_wrappers.py:1013-1034: a = new item id, percent of air cells */
    NGW_RESET_REPLACE = 3,     /* novelty_wrappers.py:1126-1148: a = item to replace, b = replacement */
    NGW_RESET_INVSET = 4,      /* novelty_wrappers.py:33,460,668-671: inventory[a] = lo */
    NGW_RESET_TREETAP = 5      /* pogostick_v0_env.py:155-178: a = tree_tap id, b = tree_log id; one tap next to a random log */
};

typedef struct {
    uint8_t op;                        /* enum ngw_op */
    uint8_t arg;
    uint8_t variant;                   /* enum ngw_break_variant for NGW_OP_BREAK */
    uint8_t reserved;
    uint8_t layers[NGW_MAX_LAYERS];    /* enum ngw_layer, outermost first, NGW_LAYER_END terminated */
} ngw_action_entry;

typedef struct {
    uint8_t n_inputs;
    uint8_t in_item[NGW_MAX_RECIPE_INPUTS];
    uint8_t in_qty[NGW_MAX_RECIPE_INPUTS];
    uint8_t out_item;
    uint8_t out_qty;
    uint8_t needs_table;               /* len(recipe['input']) > 1 (pogostick_v1_env.py:444) */
    int32_t reward_ok;                 /* 10 in Pogostick (pogostick_v1_env.py:455), 50 in Bow-v1 (bow_v1_env.py:424) */
    float cost_missing;                /* pogostick_v1_env.py:433-436 */
    float cost_no_table;               /* pogostick_v1_env.py:447-450, novelty_wrappers.py:409-410 */
    float cost_ok;                     /* pogostick_v1_env.py:463-470, novelty_wrappers.py:431-432 */
} ngw_recipe;

typedef struct {
    uint8_t kind;                      /* enum ngw_reset_kind */
    uint8_t a;
    uint8_t b;
    uint8_t lo;                        /* np.random.randint(low=lo, high=hi) percent range, hi exclusive */
    uint8_t hi;
    uint8_t reserved[3];
} ngw_reset_op;

typedef struct {
    /* ---- tables of the base env after all wrapper constructors ran ---- */
    int32_t n_items;                   /* item ids 0..n_items-1, air = 0 (pogostick_v1_env.py:200-212) */
    int32_t n_actions;                 /* external action ids 0..n_actions-1 */
    ngw_action_entry actions[NGW_MAX_ACTIONS];
    uint32_t unbreakable_mask;         /* bit i: item id i in unbreakable_items (pogostick_v1_env.py:41, novelty_wrappers.py:1116) */
    uint32_t entity_mask;              /* bit i: item id i in entities (pogostick_v1_env.py:47,538-554) */
    uint32_t break_reward_mask;        /* bit i: base Break of item i earns reward_intermediate: tree_log in the v1 envs
                                          (pogostick_v1_env.py:288), stick/plank resp. stick/string in v0
                                          (pogostick_v0_env.py:312, bow_v0_env.py:286) */
    uint32_t reserved_mask;
    uint8_t id_wall, id_crafting_table, id_tree_log, id_tree_tap, id_rubber, id_wool, id_string, id_goal;
    uint8_t id_wooden_axe, id_iron_axe; /* ids of the literal names compared at novelty_wrappers.py:56,67 */
    uint8_t id_fence;                  /* FenceRestriction.env2.fence_name (novelty_wrappers.py:928) */
    uint8_t id_fire_wall;              /* novelty_wrappers.py:1174 */
    uint8_t id_crate;                  /* novelty_wrappers.py:1085 */
    uint8_t reserved0[3];
    uint8_t crate_add[NGW_MAX_ITEMS];  /* multiset Crate.crate_ingredients as per-item counts (novelty_wrappers.py:1064-1069) */
    int32_t reward_intermediate;       /* pogostick_v1_env.py:81 */
    int32_t reward_done;               /* pogostick_v1_env.py:82 */
    int32_t reward_firewall;           /* -reward_done // 2 (novelty_wrappers.py:1187) */
    int32_t n_recipes;
    ngw_recipe recipes[NGW_MAX_RECIPES];

    /* ---- LidarInFront (observation_wrappers.py:16-80); n_beams == 0 => no lidar wrapper, obs_dim 0 ---- */
    int32_t n_beams;
    int32_t max_range;                 /* int(sqrt(2 (ms-2)^2)) at wrap time (observation_wrappers.py:25) */
    int32_t n_lidar_items;
    int8_t lidar_slot[NGW_MAX_ITEMS];  /* item id -> 0-based lidar slot, -1 = occludes but is not reported */
    int32_t n_inv_obs;
    uint8_t inv_obs_item[NGW_MAX_ITEMS]; /* item ids in sorted-name order minus unbreakables (observation_wrappers.py:77-78) */
    const int8_t* beam_lut;            /* HOST pointer, int8 [4 facings][n_beams][max_range][2] = (d_row, d_col) at sample k+1,
                                          generated with the reference's own NumPy expression (observation_wrappers.py:39-55) */

    /* ---- reset program (pogostick_v1_env.py:86-181 + novelty reset overrides) ---- */
    int32_t n_place;
    uint8_t place_item[NGW_MAX_PLACE]; /* items_quantity in insertion order (pogostick_v1_env.py:147) */
    uint8_t place_qty[NGW_MAX_PLACE];
    int32_t n_reset_ops;
    ngw_reset_op reset_ops[NGW_MAX_RESET_OPS];
    int32_t reset_obs_after_ops;       /* how many reset ops have run when the reset observation is taken (quirk Q3) */
} ngw_config;

/* info['message'] as a 16-bit code: low 5 bits = enum ngw_msg, high 11 bits = argument (item id, or for MISSING the
 * recipe slot in bits 0-2 and a mask of the missing ingredients, by recipe input position, in bits 3-6).
 * The host layer formats the reference's strings lazily (runtime.decode_message). */
enum ngw_msg {
    NGW_MSG_NONE = 0,
    NGW_MSG_BLOCK_IN_PATH = 1,        /* pogostick_v1_env.py:255, novelty_wrappers.py:1380 */
    NGW_MSG_CANNOT_BREAK = 2,         /* "Cannot break <item>" pogostick_v1_env.py:292, novelty_wrappers.py:84,958 */
    NGW_MSG_TAP_PLACED = 3,           /* pogostick_v1_env.py:301 */
    NGW_MSG_BLOCK_EXISTS = 4,         /* "Block <item> already exists when trying to place block" pogostick_v1_env.py:309 */
    NGW_MSG_NOT_IN_INVENTORY = 5,     /* pogostick_v1_env.py:312,347 */
    NGW_MSG_NO_LOG_NEAR_TAP = 6,      /* pogostick_v1_env.py:328 */
    NGW_MSG_NO_TAP = 7,               /* pogostick_v1_env.py:331 */
    NGW_MSG_NO_WOOL = 8,              /* bow_v1_env.py:304 */
    NGW_MSG_MISSING = 9,              /* "Missing items: 2 plank, 1 stick" pogostick_v1_env.py:432-440 */
    NGW_MSG_NEED_TABLE = 10,          /* pogostick_v1_env.py:452 */
    NGW_MSG_CRAFTED = 11,             /* "Crafted <item>" pogostick_v1_env.py:472 */
    NGW_MSG_NEED_AXE = 12,            /* "Cannot break without <axe> selected" novelty_wrappers.py:501 */
    NGW_MSG_CANNOT_CHOP = 13,         /* novelty_wrappers.py:1307 */
    NGW_MSG_FENCE_RESTRICTION = 14,   /* novelty_wrappers.py:955 */
    NGW_MSG_FIRE_WALL = 15            /* novelty_wrappers.py:1189 */
};

/* per-env error flags (ngw_error_flags) */
#define NGW_ERR_INVALID_ACTION 1u      /* AssertionError wrappers.py:76 / ValueError pogostick_v1_env.py:236 */
#define NGW_ERR_PLACEMENT 2u           /* AssertionError "Cannot place items, increase map size!" pogostick_v1_env.py:167 */

/* index of the counters returned by ngw_stats */
enum { NGW_STAT_STEPS = 0, NGW_STAT_EPISODES = 1, NGW_STAT_SUCCESSES = 2, NGW_STAT_REWARD_SUM = 3,
       NGW_STAT_COST_SUM = 4, NGW_STAT_RESETS = 5, NGW_STAT_INVALID = 6, NGW_STAT_RESERVED = 7, NGW_STAT_COUNT = 8 };

/* Observation row layouts (ngw_set_obs_format).  All three carry the reference's vector (observation_wrappers.py:70-80):
 * L*B lidar ranges (beam-major, L lidar items per beam) followed by the I_obs inventory quantities.
 *   NGW_OBS_I32 (default): int32 [L*B + I_obs]                         row = 4 * obs_dim bytes
 *   NGW_OBS_U8           : uint8 [L*B], zero padding to a multiple of 4, int32 [I_obs]
 *                          (a range is <= max_beam_range <= 90, so the byte is exact; inventory counts are unbounded
 *                          (quirk Q8) and stay int32).  C2: 56 + 28 = 84 bytes instead of 252.
 *   NGW_OBS_HITS         : uint8 [B][2], zero padding to a multiple of 4, int32 [I_obs]
 *                          A beam stops at the first non-air cell, so it has at most one nonzero entry among its L.  Pair b
 *                          (beam order of the vector's beam-major blocks) is (item, range): item = the reference's
 *                          lidar_items_id value 1..L (lidar slot + 1), range = the 1-based sample index the vector holds;
 *                          (0, 0) when the beam reports nothing.  vec[b*L + item - 1] = range wherever item != 0.
 *                          C2: 16 + 28 = 44 bytes.
 * Row bytes are the maximum over the batch's configs; each env's row is laid out with its own config's L, B and I_obs. */
enum { NGW_OBS_I32 = 0, NGW_OBS_U8 = 1, NGW_OBS_HITS = 2 };

/* raw device pointers of the struct-of-arrays state owned by a handle (get_observation's live references) */
typedef struct {
    int8_t*  map;        /* [n_envs_padded][map_size*map_size] item ids */
    uint8_t* pose;       /* [n_envs_padded][4] = row, col, facing id, selected item id (0 = '') */
    int32_t* inventory;  /* [n_envs_padded][inv_stride] quantity by item id */
    uint8_t* cfg_id;     /* [n_envs_padded] */
    uint32_t* episode;   /* [n_envs_padded] episode index (Philox counter word) */
    int32_t* ep_len;     /* [n_envs_padded] steps taken in the current episode */
    uint32_t* error_flags; /* [n_envs_padded] */
    int32_t inv_stride;
    int32_t obs_dim;     /* row length of the lidar observation = max over configs of L*B + I_obs */
    int64_t n_envs;
    int64_t n_envs_padded;
    int32_t map_size;
    int32_t n_configs;
    int32_t obs_format;  /* NGW_OBS_I32 / NGW_OBS_U8 / NGW_OBS_HITS */
    int32_t obs_row_bytes; /* bytes per env of the observation buffers handed to ngw_step / ngw_reset / ngw_observe */
} ngw_state_view;

typedef struct ngw_handle ngw_handle;

/* Create a batch of n_envs environments on `device` sharing one map_size and n_cfgs configs.
 * first_env_gid = global id of env 0 of this shard (Philox counters are keyed by global id, so a
 * 1/2/4/8-GPU sharding of the same job generates identical episodes). */
int ngw_create(ngw_handle** out, const ngw_config* cfgs, int32_t n_cfgs, int64_t n_envs, int32_t map_size,
               int32_t device, int64_t first_env_gid, uint64_t seed);
void ngw_destroy(ngw_handle* h);
const char* ngw_last_error(void);
int ngw_abi_version(void);

int ngw_state(ngw_handle* h, ngw_state_view* out);

/* Choose the observation row layout for every following call (default NGW_OBS_I32).  The observation pointers of
 * ngw_step / ngw_step_host / ngw_reset / ngw_observe / ngw_rollout then address rows of ngw_state_view.obs_row_bytes
 * bytes.  NGW_OBS_U8 cuts the device-to-host traffic of the host-buffer path from 266 to 94 bytes per env-step on C2,
 * NGW_OBS_HITS to 54.  ngw_rollout_policy needs NGW_OBS_I32. */
int ngw_set_obs_format(ngw_handle* h, int32_t format);

/* Which LidarInFront path the kernels take for this config on this map size (no GPU needed): 0 no lidar wrapper,
 * 1 generic LUT walk (beam count != 8), 2 factorised pointer walk, 3 line gather (the reference's 8-beam geometry). */
int ngw_lidar_path(const ngw_config* cfg, int32_t map_size);

/* cfg_id: DEVICE int32[n_envs] (NULL = all zero). */
int ngw_set_env_configs(ngw_handle* h, const int32_t* cfg_id_dev, void* stream);

/* Load `count` env states starting at env `first` from DEVICE arrays: map int8[count][ms*ms],
 * pose uint8[count][4], inventory int32[count][inv_stride]. */
int ngw_load_state(ngw_handle* h, const int8_t* map, const uint8_t* pose, const int32_t* inventory,
                   int64_t first, int64_t count, void* stream);

/* The inverse: copy `count` env states starting at env `first` out of the batch, same layouts; NULL skips an array.
 * Destinations may be device or host memory (asynchronous on `stream`; synchronize it before reading host memory). */
int ngw_export_state(ngw_handle* h, int8_t* map, uint8_t* pose, int32_t* inventory, int64_t first, int64_t count,
                     void* stream);

/* The generator every regeneration of this handle draws its maps from: ngw_reset, the auto-resets of ngw_step /
 * ngw_step_many / the host-buffer path, and the in-kernel resets of ngw_rollout / ngw_rollout_policy.
 *   NGW_RNG_PHILOX (default): counter-based, keyed by (seed, global env id, episode); the reference's distribution, not
 *                  its stream.  Setting it frees the np.random states.
 *   NGW_RNG_NUMPY: the reference's own stream.  Allocates one legacy np.random (MT19937) state per env (2.5 KB) and seeds
 *                  env e exactly as np.random.seed(seed + first_env_gid + e) does (init_genrand, pos = 624), so sharding
 *                  does not change the episodes.  Calling it again re-seeds.  Every reset then draws what the reference's
 *                  reset draws under that state, in its order, and leaves the state where the reference leaves it, so the
 *                  env's episodes continue the stream as consecutive reference resets do.  The only difference: a TREETAP
 *                  reset op (v0 envs) whose logs have no free neighbour makes the reference retry forever; here it gives up
 *                  after 2^20 attempts with NGW_ERR_PLACEMENT.  A reset that fails skips the rest of its program, as the
 *                  reference's AssertionError does.  Fails, and enqueues nothing, if seed + first_env_gid + n_envs - 1
 *                  >= 2^32.  The random policy of ngw_rollout keeps drawing from Philox (it picks actions, not maps).
 * The states are handle state: only this handle's own launches read or write them. */
enum { NGW_RNG_PHILOX = 0, NGW_RNG_NUMPY = 1 };
int ngw_set_reset_rng(ngw_handle* h, int32_t kind, void* stream);

/* The np.random states of envs [first, first + count) of a NGW_RNG_NUMPY handle in numpy's get_state() layout:
 * key uint32 [count][624], pos int32 [count].  Load reads DEVICE memory; it reads pos back to check it (a synchronising
 * copy, so not inside a stream capture).  Export writes device or host memory (asynchronous on `stream`).  A handle
 * without np.random states, a range outside the batch, or a pos outside [0, 624] fails with a message and enqueues
 * nothing. */
int ngw_load_rng_state(ngw_handle* h, const uint32_t* key, const int32_t* pos, int64_t first, int64_t count, void* stream);
int ngw_export_rng_state(ngw_handle* h, uint32_t* key, int32_t* pos, int64_t first, int64_t count, void* stream);

/* Reset envs whose mask byte is non-zero (mask DEVICE uint8[n_envs], NULL = all) with the handle's map generator
 * (ngw_set_reset_rng: Philox by default); obs (DEVICE rows of obs_row_bytes, NULL = skip) receives the reset observation
 * of the reset envs, taken after cfg.reset_obs_after_ops ops as the reference does. */
int ngw_reset(ngw_handle* h, const uint8_t* mask, void* obs, void* stream);

/* One fused step of every env: action semantics + novelties + reward/done/step_cost + LidarInFront
 * observation (+ Philox auto-reset of done envs when auto_reset != 0 — queued by the step kernel and regenerated by
 * a second small kernel of the same call; the observation row of a regenerated env is the new episode's reset
 * observation, taken after cfg.reset_obs_after_ops ops like ngw_reset —, + truncation when max_episode_steps > 0).
 * All pointers are DEVICE pointers, obs = [n_envs] rows of obs_row_bytes (int32 [n_envs][obs_dim] by default),
 * 16-byte aligned; obs may be NULL when obs_dim == 0. */
int ngw_step(ngw_handle* h, const int32_t* actions, void* obs, float* reward, uint8_t* done,
             float* step_cost, uint8_t* result, int32_t auto_reset, int32_t max_episode_steps, void* stream);

/* Several handles stepped by ONE call, in the order given, on one stream (the loop over env pools a driver would write
 * around ngw_step, tests/random_action.py:51-55 per pool).  The library issues the launches back to back, so it knows
 * that nothing sits between them: consecutive items that step different handles and share no caller buffer overlap
 * exactly as consecutive ngw_step calls do inside a stream capture (see ngw_concurrent_launch_count) — in eager mode too.
 * The caller must not enqueue work on `stream` from another thread during the call.  Pointers as in ngw_step. */
typedef struct ngw_step_item {
    ngw_handle* h;
    const int32_t* actions;
    void* obs;
    float* reward;
    uint8_t* done;
    float* step_cost;
    uint8_t* result;
} ngw_step_item;
int ngw_step_many(const ngw_step_item* items, int32_t n_items, int32_t auto_reset, int32_t max_episode_steps, void* stream);

/* Optional: DEVICE uint16[n_envs] that every following ngw_step / ngw_rollout fills with the step's message code
 * (NULL switches it off again; off by default — the hot path then writes nothing). */
int ngw_set_message_buffer(ngw_handle* h, uint16_t* msg_dev);

/* Optional episode-end outputs of the one-step calls (ngw_step, ngw_step_many, ngw_step_host, _begin/_end), what a learner
 * needs to bootstrap at a time limit (gym 0.18's info['TimeLimit.truncated'], and the last observation of an episode that
 * the auto-reset replaced).  Each pointer may be NULL, which switches that output off; both are off by default.
 *   truncated_dev: DEVICE uint8[n_envs].  Every valid env of a call gets 1 when this step reached max_episode_steps and the
 *                  env's own step did not end the episode (gym's TimeLimit rule), else 0; invalid-action lanes get 0.
 *                  done == terminated | truncated, the two disjoint: an env that terminates on the limit's step reports
 *                  terminated.  Without auto_reset an env past the limit reports done, and so truncated, on every step.
 *   final_obs_dev: DEVICE rows of obs_row_bytes in the handle's layout, 16-byte aligned.  Row e is written only for the
 *                  envs this call's auto-reset regenerated: the observation the step produced, byte for byte what obs
 *                  would hold without auto_reset, before the new episode's reset observation replaced it.  Other rows
 *                  are left untouched.  Ignored without a LidarInFront observation (obs_dim == 0) or an obs buffer.
 * The host-buffer path writes the same DEVICE buffers on the handle's stream (valid once ngw_step_host / _end returned).
 * ngw_observe, ngw_reset, ngw_rollout and ngw_rollout_policy never touch either buffer. */
int ngw_set_episode_end_buffers(ngw_handle* h, uint8_t* truncated_dev, void* final_obs_dev);

/* Optional per-step record of the K-step rollouts (ngw_rollout, ngw_rollout_policy): while it is set, a rollout of n_steps
 * fills, for every step t < n_steps and env e < n_envs, element [t][e] of each non-NULL buffer with what n_steps single
 * ngw_step calls would report at their t-th step (same seed, state, actions, auto_reset and max_episode_steps, episode-end
 * buffers on).  Every buffer is DEVICE memory laid out [max_steps][n_envs_padded] (ngw_state_view.n_envs_padded: each
 * step's block starts on a 128-byte boundary; what padding elements hold is unspecified).
 *   obs       rows of obs_row_bytes in the observation format in force at launch, 16-byte aligned: the observation of
 *             env e after step t and its auto-reset, observed after ALL of the reset ops — what ngw_observe returns right
 *             after the t-th ngw_step, and what the rollout's policy acts on at step t + 1 (so obs[n_steps - 1] equals the
 *             rollout's obs output).  It differs from ngw_step's obs row only for an env regenerated at step t under a
 *             config with reset_obs_after_ops < n_reset_ops.
 *   reward, step_cost, done, result   as ngw_step's outputs (step_cost bit for bit; no summation).
 *   truncated 1 where step t reached max_episode_steps and the env's own step did not end the episode (gym's TimeLimit
 *             rule, as ngw_set_episode_end_buffers); 0 on invalid-action lanes.
 *   final_obs rows like obs, written ONLY where step t's auto-reset regenerated env e: the observation the step produced,
 *             before the reset.  Every other row is left untouched.
 * Invalid actions record zeros and the observation of the unchanged state, as ngw_step does.  obs / final_obs are ignored
 * without a LidarInFront observation (obs_dim == 0).  A rollout with n_steps > max_steps fails and enqueues nothing.
 * Everything a rollout returns without a record is bit-identical with one.  ngw_step, ngw_step_many, the host-buffer path,
 * ngw_observe and ngw_reset never touch the record.  The buffers are the caller's; the handle keeps the pointers. */
typedef struct ngw_rollout_record {
    int32_t max_steps;      /* steps the buffers hold (>= 1) */
    void* obs;              /* rows of obs_row_bytes, [max_steps][n_envs_padded], 16-byte aligned; NULL = skip */
    float* reward;          /* [max_steps][n_envs_padded]; NULL = skip (same for every field below) */
    float* step_cost;
    uint8_t* done;
    uint8_t* result;
    uint8_t* truncated;
    void* final_obs;        /* rows like obs, 16-byte aligned; written only for envs regenerated at step t */
} ngw_rollout_record;
/* rec is copied; NULL switches the record off (the default).  Fails on misaligned pointers or max_steps < 1. */
int ngw_set_rollout_record(ngw_handle* h, const ngw_rollout_record* rec);

/* Same call with HOST buffers (the reference-facing path): copies actions in (H2D), steps, copies
 * obs/reward/done/step_cost/result out (D2H) on the handle's own stream; returns after the outputs are valid
 * on the host.  The step is ordered after everything earlier calls on this handle enqueued on the caller's streams
 * (ngw_reset, ngw_load_state, ngw_step ...), and later device-path calls wait for it.  Pinned buffers make the copies true DMA; if step_cost == reward + n, done == step_cost + n and
 * result == done + n (bytes: reward | step_cost | done | result contiguous) the four small outputs travel in one copy;
 * if moreover reward == (char*)obs + round_up(n_envs * obs_row_bytes, 16) — one block: observation rows | pad to 16 |
 * reward | step_cost | done | result — the WHOLE step travels in one copy. */
int ngw_step_host(ngw_handle* h, const int32_t* actions, void* obs, float* reward, uint8_t* done,
                  float* step_cost, uint8_t* result, int32_t auto_reset, int32_t max_episode_steps);

/* K-step rollout in ONE launch (SURVEY §8f N1): every tile stays in shared memory for n_steps consecutive steps.
 * actions: DEVICE int32[n_steps][n_envs], or NULL = uniform random policy drawn on the device with Philox
 * (policy_seed, global env id, step index / 4: one block serves four steps; exact uniformity by multiply-shift with
 * rejection) — the tests/random_action.py loop without the host.  reward_sum / cost_sum
 * accumulate over the steps, done_count counts finished episodes, last_done / last_result are the final step's, obs is
 * the observation after the last step; actions_out (DEVICE int32[n_steps][n_envs], NULL = skip) records the actions.
 * ngw_set_rollout_record adds the per-step transitions (observation, reward, done, truncation, terminal observation). */
int ngw_rollout(ngw_handle* h, const int32_t* actions, int32_t n_steps, uint64_t policy_seed, void* obs,
                float* reward_sum, float* cost_sum, int32_t* done_count, uint8_t* last_done, uint8_t* last_result,
                int32_t* actions_out, int32_t auto_reset, int32_t max_episode_steps, void* stream);

/* Closed-loop K-step rollout: at every step the action is argmax_a (bias[a] + sum_j obs[j] * weights[j][a]) over the
 * env's valid action ids, computed on the device from the current LidarInFront observation (lowest id wins ties).
 * weights: DEVICE int32[obs_dim][n_policy_actions], bias: DEVICE int32[n_policy_actions], n_policy_actions <= 16.
 * Integer arithmetic => bit-reproducible on the host.  Outputs as ngw_rollout.  Needs NGW_OBS_I32 rows.  With auto_reset,
 * an env regenerated inside a rollout is observed after ALL of its reset ops (the next step needs the final state); the
 * per-step record (ngw_set_rollout_record) holds the observations the policy acted on. */
int ngw_rollout_policy(ngw_handle* h, const int32_t* weights, const int32_t* bias, int32_t n_policy_actions,
                       int32_t n_steps, void* obs, float* reward_sum, float* cost_sum, int32_t* done_count,
                       uint8_t* last_done, uint8_t* last_result, int32_t* actions_out, int32_t auto_reset,
                       int32_t max_episode_steps, void* stream);

/* The host-buffer step split in two, so that a caller with several batches can keep PCIe busy: _begin enqueues the
 * H2D copy, the launch and the D2H copies on the handle's own stream and returns; _end blocks until this handle's
 * outputs are valid on the host.  ngw_step_host == _begin + _end. */
int ngw_step_host_begin(ngw_handle* h, const int32_t* actions, void* obs, float* reward, uint8_t* done,
                        float* step_cost, uint8_t* result, int32_t auto_reset, int32_t max_episode_steps);
int ngw_step_host_end(ngw_handle* h);

/* LidarInFront.observation of the current state into DEVICE [n_envs] rows of obs_row_bytes. */
int ngw_observe(ngw_handle* h, void* obs, void* stream);

/* AgentMap.get_agentView (observation_wrappers.py:98-118): the (2*view+1)^2 zero-padded crop of the grid centred on the
 * agent, DEVICE int8[n_envs][2*view+1][2*view+1]. */
int ngw_agent_map(ngw_handle* h, int8_t* out, int32_t view, void* stream);

/* Copy the NGW_STAT_COUNT accumulated counters (doubles) to DEVICE out8; reset_after != 0 zeroes them. */
int ngw_stats(ngw_handle* h, double* out8_dev, int32_t reset_after, void* stream);

/* Number of kernel launches issued by this handle so far (bench.py's gpu_launches claim). */
int64_t ngw_launch_count(ngw_handle* h);

/* Of those, the one-step launches that ran OVERLAPPED with their predecessor.  Two consecutive ngw_step launches on one
 * stream are independent when they step different handles and share no caller buffer (actions, observations, reward,
 * done, step_cost, result, messages); the library overlaps them only when it can PROVE that nothing was enqueued between
 * them, which it can inside a stream capture (the stream's dependency set is exactly the previous launch's graph node):
 * the tile warps of the second launch then do not wait for the first grid, while one gate warp per CTA does and only
 * then lets the third launch start — at most two launches are in flight, completion stays in stream order, results are
 * identical.  Single eager ngw_step calls always wait (ngw_step_many carries the same proof without a capture).
 * NGW_NO_CONCURRENT=1 (read by ngw_create) turns the overlap off. */
int64_t ngw_concurrent_launch_count(ngw_handle* h);

#ifdef __cplusplus
}
#endif
#endif /* NGW_H */
