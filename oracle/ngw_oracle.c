/*
 * ngw_oracle.c — CPU restatement of the reference's NovelGridworld step / reset / LidarInFront path, and (last section)
 * of the DEVICE's Philox map generator and random policy, which by design share the reference's distribution but not
 * its stream.
 *
 * TEST INFRASTRUCTURE, NOT PRODUCT.  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
 * --impl reference legs may load this library; the product (gym_novel_gridworlds_b200) never does and
 * has no CPU fallback.
 *
 * Parity is PINNED: tests/golden/ *.npz hold traces produced by running the UNMODIFIED reference
 * (/root/reference/gym_novel_gridworlds, through oracle/gymstub) with oracle/gen_golden.py; the CPU
 * suite replays every trace through this file (tests/test_oracle_golden.py), including the reference's
 * reset states, which this file regenerates bit-for-bit from the seed by restating the legacy
 * np.random (MT19937) draw sequence.
 *
 * Reference files restated (paths relative to /root/reference/gym_novel_gridworlds):
 *   envs/pogostick_v1_env.py:86-181   reset, add_item_to_map
 *   envs/pogostick_v1_env.py:230-367  step            envs/bow_v1_env.py:228-340 (Extract_string)
 *   envs/pogostick_v1_env.py:369-474  update_block_in_front, is_block_in_front_next_to, craft
 *   envs/pogostick_v1_env.py:524-554  add_fence_around, grab_entities
 *   observation_wrappers.py:32-80     LidarInFront.get_lidarSignal / observation
 *   novelty_wrappers.py               every step()/reset() override; cited at each function
 * The wrapper chain itself arrives flattened as an `ngw_config` (include/ngw.h); recursion over
 * `layers` below plays the role of the reference's nested `self.env.step(action_id)` calls.
 *
 * NumPy (any version with the legacy RandomState; README pins 1.19.4) algorithms restated:
 *   RandomState.seed(int)            -> init_genrand
 *   randint / choice(n, size=1)      -> masked rejection on 32-bit outputs (legacy _bounded_uint64, rng <= 2^32-1)
 *   shuffle                          -> Fisher-Yates from the top, j = random_interval(i)
 */
#include "../include/ngw.h"

#include <math.h>
#include <pthread.h>
#include <stdlib.h>
#include <string.h>

/* ------------------------------------------------------------------ MT19937 (legacy np.random) */
typedef struct {
    uint32_t key[624];
    int pos;
} ngo_mt;

void ngo_mt_seed(ngo_mt* s, uint32_t seed) {
    for (int i = 0; i < 624; i++) {
        s->key[i] = seed;
        seed = 1812433253u * (seed ^ (seed >> 30)) + (uint32_t)i + 1u;
    }
    s->pos = 624;
}

static void mt_refill(ngo_mt* s) {
    const uint32_t UPPER = 0x80000000u, LOWER = 0x7fffffffu, MAGIC = 0x9908b0dfu;
    uint32_t* k = s->key;
    int i;
    for (i = 0; i < 624 - 397; i++) {
        uint32_t y = (k[i] & UPPER) | (k[i + 1] & LOWER);
        k[i] = k[i + 397] ^ (y >> 1) ^ ((y & 1u) ? MAGIC : 0u);
    }
    for (; i < 623; i++) {
        uint32_t y = (k[i] & UPPER) | (k[i + 1] & LOWER);
        k[i] = k[i + (397 - 624)] ^ (y >> 1) ^ ((y & 1u) ? MAGIC : 0u);
    }
    uint32_t y = (k[623] & UPPER) | (k[0] & LOWER);
    k[623] = k[396] ^ (y >> 1) ^ ((y & 1u) ? MAGIC : 0u);
    s->pos = 0;
}

uint32_t ngo_mt_next(ngo_mt* s) {
    if (s->pos == 624) mt_refill(s);
    uint32_t y = s->key[s->pos++];
    y ^= (y >> 11);
    y ^= (y << 7) & 0x9d2c5680u;
    y ^= (y << 15) & 0xefc60000u;
    y ^= (y >> 18);
    return y;
}

/* uniform integer in [0, max] — shared core of legacy randint / choice / shuffle */
static uint32_t mt_interval(ngo_mt* s, uint32_t max) {
    if (max == 0) return 0;
    uint32_t mask = max;
    mask |= mask >> 1; mask |= mask >> 2; mask |= mask >> 4; mask |= mask >> 8; mask |= mask >> 16;
    uint32_t v;
    do { v = ngo_mt_next(s) & mask; } while (v > max);
    return v;
}

/* np.random.randint(low, high, size=1)[0] / np.random.choice(n, size=1)[0] */
uint32_t ngo_randint(ngo_mt* s, uint32_t low, uint32_t high) { return low + mt_interval(s, high - 1u - low); }

/* np.random.shuffle on a 1-d array / list of n elements */
void ngo_shuffle_i32(ngo_mt* s, int32_t* a, int n) {
    for (int i = n - 1; i >= 1; i--) {
        int j = (int)mt_interval(s, (uint32_t)i);
        int32_t t = a[i]; a[i] = a[j]; a[j] = t;
    }
}

/* ------------------------------------------------------------------ small helpers */
typedef struct {
    const ngw_config* cfg;
    int ms;
    int8_t* map;       /* [ms*ms] */
    uint8_t* pose;     /* r, c, facing, selected */
    int32_t* inv;      /* by item id */
} env_t;

#define CELL(e, r, c) ((e)->map[(r) * (e)->ms + (c)])

static int in_mask(uint32_t mask, int item) { return item >= 0 && item < 32 && ((mask >> item) & 1u); }

/* update_block_in_front (pogostick_v1_env.py:369-383): N r-1, S r+1, W c-1, E c+1 */
static void front_of(const env_t* e, int* fr, int* fc) {
    int r = e->pose[0], c = e->pose[1];
    switch (e->pose[2]) {
        case NGW_NORTH: r -= 1; break;
        case NGW_SOUTH: r += 1; break;
        case NGW_WEST:  c -= 1; break;
        default:        c += 1; break;
    }
    *fr = r; *fc = c;
}

/* is_block_in_front_next_to (pogostick_v1_env.py:391-411): 4-neighbours of the FRONT cell, bounds-checked */
static int front_next_to(const env_t* e, int item) {
    int r, c;
    front_of(e, &r, &c);
    int hi = e->ms - 1;
    if (r - 1 >= 0 && r - 1 <= hi && CELL(e, r - 1, c) == item) return 1;
    if (r + 1 >= 0 && r + 1 <= hi && CELL(e, r + 1, c) == item) return 1;
    if (c - 1 >= 0 && c - 1 <= hi && CELL(e, r, c - 1) == item) return 1;
    if (c + 1 >= 0 && c + 1 <= hi && CELL(e, r, c + 1) == item) return 1;
    return 0;
}

/* grab_entities (pogostick_v1_env.py:538-554): 3x3 around the agent, row-major */
static void grab_entities(env_t* e) {
    int r = e->pose[0], c = e->pose[1];
    for (int rr = r - 1; rr <= r + 1; rr++)
        for (int cc = c - 1; cc <= c + 1; cc++) {
            int id = CELL(e, rr, cc);
            if (id != 0 && in_mask(e->cfg->entity_mask, id)) {
                CELL(e, rr, cc) = 0;
                e->inv[id] += 1;
            }
        }
}

typedef struct {
    int reward;
    int done;
    int result;
    float cost;
    int msg;           /* info['message'] as enum ngw_msg | argument << 5 (include/ngw.h) */
} out_t;

static int msg_code(int kind, int arg) { return kind | (arg << 5); }

/* the "Update after each step" block every step path ends with (pogostick_v1_env.py:349-357,
 * duplicated e.g. at novelty_wrappers.py:86-97): entities, then done / reward_done */
static void post_step(env_t* e, out_t* o) {
    grab_entities(e);
    o->done = 0;
    if (e->inv[e->cfg->id_goal] >= 1) {
        o->reward = e->cfg->reward_done;
        o->done = 1;
    }
}

/* craft (pogostick_v1_env.py:413-474, bow_v1_env.py:386-441, novelty_wrappers.py:371-436) */
static void craft(env_t* e, const ngw_recipe* rc, out_t* o) {
    o->reward = -1; o->result = 1; o->cost = 0.0f;
    int missing = 0;                             /* "Missing items: ..." lists the short inputs in recipe order */
    for (int i = 0; i < rc->n_inputs; i++) {
        int item = rc->in_item[i];
        if (item == NGW_NONE || e->inv[item] < rc->in_qty[i]) missing |= 1 << i;
    }
    if (missing) {
        o->result = 0; o->cost = rc->cost_missing;
        o->msg = msg_code(NGW_MSG_MISSING, (int)(rc - e->cfg->recipes) | (missing << 3));
        return;
    }
    if (rc->needs_table) {
        int fr, fc;
        front_of(e, &fr, &fc);
        if (CELL(e, fr, fc) != e->cfg->id_crafting_table) {
            o->result = 0; o->cost = rc->cost_no_table; o->msg = NGW_MSG_NEED_TABLE; return;
        }
    }
    o->reward = rc->reward_ok;
    for (int i = 0; i < rc->n_inputs; i++) e->inv[rc->in_item[i]] -= rc->in_qty[i];
    e->inv[rc->out_item] += rc->out_qty;
    o->cost = rc->cost_ok;
    o->msg = msg_code(NGW_MSG_CRAFTED, rc->out_item);
}

/* The Break family.  Every variant starts with update_block_in_front and the unbreakable test. */
static void do_break(env_t* e, const ngw_action_entry* a, out_t* o) {
    const ngw_config* cfg = e->cfg;
    int fr, fc;
    front_of(e, &fr, &fc);
    int front = CELL(e, fr, fc);
    int sel = e->pose[3];
    o->reward = -1; o->result = 1; o->cost = 3600.0f;
    if (in_mask(cfg->unbreakable_mask, front)) { o->result = 0; o->msg = msg_code(NGW_MSG_CANNOT_BREAK, front); return; }
    switch (a->variant) {
        case NGW_BRK_BASE:                       /* pogostick_v1_env.py:283-289 */
            CELL(e, fr, fc) = 0;
            e->inv[front] += 1;
            if (in_mask(cfg->break_reward_mask, front)) o->reward = cfg->reward_intermediate;
            break;
        case NGW_BRK_AXE:
        case NGW_BRK_AXE_INC: {                  /* novelty_wrappers.py:55-81 */
            int qty = (a->variant == NGW_BRK_AXE_INC) ? 2 : 1;
            if (e->inv[a->arg] >= 1 && cfg->id_wooden_axe != NGW_NONE && sel == cfg->id_wooden_axe) {
                CELL(e, fr, fc) = 0; e->inv[front] += qty;
                o->reward = cfg->reward_intermediate; o->cost = 3600.0f * 0.5f;
            } else if (e->inv[a->arg] >= 1 && cfg->id_iron_axe != NGW_NONE && sel == cfg->id_iron_axe) {
                CELL(e, fr, fc) = 0; e->inv[front] += qty;
                o->reward = cfg->reward_intermediate; o->cost = 3600.0f * 0.25f;
            } else {                             /* no reward even for tree_log (SURVEY Q4) */
                CELL(e, fr, fc) = 0; e->inv[front] += 1;
            }
            break;
        }
        case NGW_BRK_AXETOBREAK:                 /* novelty_wrappers.py:482-501 */
            if (e->inv[a->arg] >= 1 && cfg->id_wooden_axe != NGW_NONE && sel == cfg->id_wooden_axe) {
                CELL(e, fr, fc) = 0; e->inv[front] += 1;
                o->reward = cfg->reward_intermediate; o->cost = 1800.0f;
            } else if (e->inv[a->arg] >= 1 && cfg->id_iron_axe != NGW_NONE && sel == cfg->id_iron_axe) {
                CELL(e, fr, fc) = 0; e->inv[front] += 1;
                o->reward = cfg->reward_intermediate; o->cost = 900.0f;
            } else {                             /* "Cannot break without <axe> selected" */
                o->result = 0; o->msg = msg_code(NGW_MSG_NEED_AXE, a->arg);
            }
            break;
        case NGW_BRK_INCREASE:                   /* novelty_wrappers.py:1444-1454 */
            CELL(e, fr, fc) = 0;
            e->inv[front] += (a->arg == NGW_NONE || a->arg == front) ? 2 : 1;
            o->reward = cfg->reward_intermediate;
            break;
        default: break;
    }
}

/* terminal opcode = the innermost `step` body that finally handles the action */
static void terminal_step(env_t* e, const ngw_action_entry* a, out_t* o) {
    const ngw_config* cfg = e->cfg;
    int r = e->pose[0], c = e->pose[1], f = e->pose[2];
    int fr, fc;
    front_of(e, &fr, &fc);
    o->reward = -1; o->result = 1; o->cost = 0.0f; o->done = 0; o->msg = NGW_MSG_NONE;   /* pogostick_v1_env.py:239-242 */
    switch (a->op) {
        case NGW_OP_NOOP: break;
        case NGW_OP_FORWARD:                      /* pogostick_v1_env.py:244-257 */
            if (CELL(e, fr, fc) == 0) { e->pose[0] = (uint8_t)fr; e->pose[1] = (uint8_t)fc; }
            else { o->result = 0; o->msg = NGW_MSG_BLOCK_IN_PATH; }
            o->cost = 27.906975f;
            break;
        case NGW_OP_LEFT: {                       /* pogostick_v1_env.py:258-268: N->W, S->E, W->S, E->N */
            static const uint8_t left[4] = {NGW_WEST, NGW_EAST, NGW_SOUTH, NGW_NORTH};
            e->pose[2] = left[f]; o->cost = 24.0f; break;
        }
        case NGW_OP_RIGHT: {                      /* pogostick_v1_env.py:269-279: N->E, S->W, W->N, E->S */
            static const uint8_t right[4] = {NGW_EAST, NGW_WEST, NGW_NORTH, NGW_SOUTH};
            e->pose[2] = right[f]; o->cost = 24.0f; break;
        }
        case NGW_OP_BREAK: do_break(e, a, o); break;
        case NGW_OP_PLACE_TREE_TAP:               /* pogostick_v1_env.py:295-314 */
            if (e->inv[cfg->id_tree_tap] >= 1) {
                if (CELL(e, fr, fc) == 0) {
                    CELL(e, fr, fc) = (int8_t)cfg->id_tree_tap;
                    e->inv[cfg->id_tree_tap] -= 1;
                    if (front_next_to(e, cfg->id_tree_log)) o->reward = cfg->reward_intermediate;
                    o->msg = NGW_MSG_TAP_PLACED;
                } else { o->result = 0; o->msg = msg_code(NGW_MSG_BLOCK_EXISTS, CELL(e, fr, fc)); }
            } else { o->result = 0; o->msg = NGW_MSG_NOT_IN_INVENTORY; }
            o->cost = 300.0f;
            break;
        case NGW_OP_EXTRACT_RUBBER:               /* pogostick_v1_env.py:315-331, novelty_wrappers.py:1537-1551 */
            o->cost = 120.0f;
            if (CELL(e, fr, fc) == cfg->id_tree_tap) {
                if (front_next_to(e, cfg->id_tree_log)) {
                    e->inv[cfg->id_rubber] += a->arg;
                    o->reward = cfg->reward_intermediate; o->cost = 50000.0f;
                } else { o->result = 0; o->msg = NGW_MSG_NO_LOG_NEAR_TAP; }
            } else { o->result = 0; o->msg = NGW_MSG_NO_TAP; }
            break;
        case NGW_OP_EXTRACT_STRING:               /* bow_v1_env.py:293-304, novelty_wrappers.py:1524-1536 */
            o->cost = 120.0f;
            if (CELL(e, fr, fc) == cfg->id_wool) {
                e->inv[cfg->id_string] += a->arg;
                CELL(e, fr, fc) = 0;
                o->reward = cfg->reward_intermediate; o->cost = 5000.0f;
            } else { o->result = 0; o->msg = NGW_MSG_NO_WOOL; }
            break;
        case NGW_OP_CRAFT: craft(e, &cfg->recipes[a->arg], o); break;
        case NGW_OP_SELECT:                       /* pogostick_v1_env.py:338-347 */
            o->cost = 120.0f;
            if (a->arg != NGW_NONE && e->inv[a->arg] >= 1) e->pose[3] = a->arg;
            else { o->result = 0; o->msg = NGW_MSG_NOT_IN_INVENTORY; }
            break;
        case NGW_OP_CHOP: {                       /* novelty_wrappers.py:1291-1307 */
            int front = CELL(e, fr, fc);
            o->cost = 3600.0f * 1.2f;
            if (!in_mask(cfg->unbreakable_mask, front)) {
                CELL(e, fr, fc) = 0; e->inv[front] += 2; o->reward = cfg->reward_intermediate;
            } else { o->result = 0; o->msg = msg_code(NGW_MSG_CANNOT_CHOP, front); }
            break;
        }
        case NGW_OP_JUMP: {                       /* novelty_wrappers.py:1363-1382: 2 ahead, middle cell ignored */
            int tr = r + 2 * (fr - r), tc = c + 2 * (fc - c);
            if (tr >= 0 && tr <= e->ms - 1 && tc >= 0 && tc <= e->ms - 1 && CELL(e, tr, tc) == 0) {
                e->pose[0] = (uint8_t)tr; e->pose[1] = (uint8_t)tc;
            } else { o->result = 0; o->msg = NGW_MSG_BLOCK_IN_PATH; }
            o->cost = 27.906975f * 2.0f;
            break;
        }
        default: break;
    }
    post_step(e, o);
}

/* layered_step(i): the i-th pass-through wrapper's step(), calling "self.env.step" = layered_step(i+1) */
static void layered_step(env_t* e, const ngw_action_entry* a, int i, out_t* o) {
    const ngw_config* cfg = e->cfg;
    int layer = (i < NGW_MAX_LAYERS) ? a->layers[i] : NGW_LAYER_END;
    if (layer == NGW_LAYER_END) { terminal_step(e, a, o); return; }
    if (layer == NGW_LAYER_CRATE) {               /* novelty_wrappers.py:1085-1090 */
        int fr, fc;
        front_of(e, &fr, &fc);
        if (CELL(e, fr, fc) == cfg->id_crate)
            for (int it = 0; it < cfg->n_items; it++) e->inv[it] += cfg->crate_add[it];
        layered_step(e, a, i + 1, o);
        return;
    }
    if (layer == NGW_LAYER_FIREWALL) {            /* novelty_wrappers.py:1169-1189 */
        layered_step(e, a, i + 1, o);
        int r = e->pose[0], c = e->pose[1], hi = e->ms - 1, fw = cfg->id_fire_wall, close_to = 0;
        if (r - 1 >= 0 && r - 1 <= hi && CELL(e, r - 1, c) == fw) close_to = 1;
        else if (r + 1 >= 0 && r + 1 <= hi && CELL(e, r + 1, c) == fw) close_to = 1;
        else if (c - 1 >= 0 && c - 1 <= hi && CELL(e, r, c - 1) == fw) close_to = 1;
        else if (c + 1 >= 0 && c + 1 <= hi && CELL(e, r, c + 1) == fw) close_to = 1;
        if (close_to) { o->reward = cfg->reward_firewall; o->done = 1; o->msg = NGW_MSG_FIRE_WALL; }
        return;
    }
    /* FenceRestriction medium / hard (novelty_wrappers.py:918-973) */
    {
        int fr, fc;
        front_of(e, &fr, &fc);
        int front = CELL(e, fr, fc), fence = cfg->id_fence;
        int result = 1, msg = NGW_MSG_NONE;
        o->reward = -1;
        if (!in_mask(cfg->unbreakable_mask, front)) {
            if (front == fence) {
                layered_step(e, a, i + 1, o);                        /* fences are always breakable */
            } else {
                int restricted = 0;
                int r = e->pose[0], c = e->pose[1], f = e->pose[2];
                if (layer == NGW_LAYER_FENCE_MEDIUM) {                /* fence left/right of the AGENT */
                    if (f == NGW_NORTH || f == NGW_SOUTH) {
                        if (CELL(e, r, c - 1) == fence || CELL(e, r, c + 1) == fence) restricted = 1;
                    } else {
                        if (CELL(e, r - 1, c) == fence || CELL(e, r + 1, c) == fence) restricted = 1;
                    }
                } else {                                              /* any fence in the 3x3 around the FRONT cell */
                    for (int rr = fr - 1; rr <= fr + 1; rr++)
                        for (int cc = fc - 1; cc <= fc + 1; cc++)
                            if (rr >= 0 && rr < e->ms && cc >= 0 && cc < e->ms && CELL(e, rr, cc) == fence)
                                restricted = 1;
                }
                if (!restricted) layered_step(e, a, i + 1, o);
                else { result = 0; msg = NGW_MSG_FENCE_RESTRICTION; }
            }
        } else { result = 0; msg = msg_code(NGW_MSG_CANNOT_BREAK, front); }
        /* the outer post block always re-runs and OVERWRITES info (SURVEY Q5, novelty_wrappers.py:960-973) */
        int reward = o->reward;
        grab_entities(e);
        o->done = 0;
        if (e->inv[cfg->id_goal] >= 1) { reward = cfg->reward_done; o->done = 1; }
        o->reward = reward; o->result = result; o->cost = 3600.0f; o->msg = msg;
    }
}

/* ------------------------------------------------------------------ public: one env step */
/* returns 0, or NGW_ERR_INVALID_ACTION (state untouched, outputs zeroed, message code 0).  msg may be NULL. */
int ngo_step(const ngw_config* cfg, int ms, int8_t* map, uint8_t* pose, int32_t* inv, int32_t action,
             float* reward, uint8_t* done, float* cost, uint8_t* result, uint16_t* msg) {
    env_t e = {cfg, ms, map, pose, inv};
    if (action < 0 || action >= cfg->n_actions || cfg->actions[action].op == NGW_OP_INVALID) {
        *reward = 0.0f; *done = 0; *cost = 0.0f; *result = 0;
        if (msg) *msg = NGW_MSG_NONE;
        return NGW_ERR_INVALID_ACTION;
    }
    out_t o = {-1, 0, 1, 0.0f, NGW_MSG_NONE};
    layered_step(&e, &cfg->actions[action], 0, &o);
    *reward = (float)o.reward; *done = (uint8_t)o.done; *cost = o.cost; *result = (uint8_t)o.result;
    if (msg) *msg = (uint16_t)o.msg;
    return 0;
}

/* ------------------------------------------------------------------ LidarInFront */
/* (d_row, d_col) of sample k (1-based) of beam b for a facing — observation_wrappers.py:39-55 in C doubles:
 * linspace(theta - pi, theta + pi, B + 1)[:-1]; np.round(x, 2) = rint(x * 100) / 100; np.round(k * x) = rint */
void ngo_beam_offset(int facing, int n_beams, int b, int k, int* d_row, int* d_col) {
    static const double PI = 3.141592653589793;
    double theta = (facing == NGW_NORTH) ? PI : (facing == NGW_SOUTH) ? 0.0 : (facing == NGW_WEST) ? 3 * PI / 2 : PI / 2;
    double start = theta - PI, stop = theta + PI;
    double step = (stop - start) / (double)n_beams;
    double angle = start + (double)b * step;
    double x = rint(cos(angle) * 100.0) / 100.0;
    double y = rint(sin(angle) * 100.0) / 100.0;
    *d_row = (int)rint((double)k * x);
    *d_col = (int)rint((double)k * y);
}

/* obs[0 .. L*B + n_inv_obs) — observation_wrappers.py:32-80.  The reference evaluates cos/sin once per beam per
 * call; the per-beam ratios depend only on (facing, n_beams), so they are cached per thread. */
void ngo_observe(const ngw_config* cfg, int ms, const int8_t* map, const uint8_t* pose, const int32_t* inv,
                 int32_t* obs) {
    static __thread int cached_beams = -1;
    static __thread double ratio[4][64][2];
    int L = cfg->n_lidar_items, B = cfg->n_beams;
    int r = pose[0], c = pose[1];
    if (B != cached_beams && B <= 64) {
        static const double PI = 3.141592653589793;
        for (int f = 0; f < 4; f++) {
            double theta = (f == NGW_NORTH) ? PI : (f == NGW_SOUTH) ? 0.0 : (f == NGW_WEST) ? 3 * PI / 2 : PI / 2;
            double start = theta - PI, step = ((theta + PI) - start) / (double)B;
            for (int b = 0; b < B; b++) {
                double angle = start + (double)b * step;
                ratio[f][b][0] = rint(cos(angle) * 100.0) / 100.0;      /* np.round(np.cos(angle), 2) */
                ratio[f][b][1] = rint(sin(angle) * 100.0) / 100.0;
            }
        }
        cached_beams = B;
    }
    for (int i = 0; i < L * B; i++) obs[i] = 0;
    for (int b = 0; b < B; b++) {
        double x, y;
        if (B <= 64) { x = ratio[pose[2]][b][0]; y = ratio[pose[2]][b][1]; }
        else {                                                        /* more beams than the cache holds: evaluate directly */
            static const double PI2 = 3.141592653589793;
            int f = pose[2];
            double theta = (f == NGW_NORTH) ? PI2 : (f == NGW_SOUTH) ? 0.0 : (f == NGW_WEST) ? 3 * PI2 / 2 : PI2 / 2;
            double start = theta - PI2, step = ((theta + PI2) - start) / (double)B;
            double angle = start + (double)b * step;
            x = rint(cos(angle) * 100.0) / 100.0;
            y = rint(sin(angle) * 100.0) / 100.0;
        }
        for (int k = 1; k <= cfg->max_range; k++) {
            int rr = r + (int)rint((double)k * x), cc = c + (int)rint((double)k * y);   /* np.round(k * ratio) */
            if (rr < 0 || rr >= ms || cc < 0 || cc >= ms) break;      /* unreachable on a walled map */
            int id = map[rr * ms + cc];
            if (id != 0) {
                int slot = cfg->lidar_slot[id];
                if (slot >= 0) obs[b * L + slot] = k;
                break;
            }
        }
    }
    for (int i = 0; i < cfg->n_inv_obs; i++) obs[L * B + i] = inv[cfg->inv_obs_item[i]];
}

/* ------------------------------------------------------------------ reset with the legacy np.random stream */
static int percent_count(int n, int pct) { return (int)ceil((double)n * ((double)pct / 100.0)); }

/* add_item_to_map (pogostick_v1_env.py:159-181) on the shrinking `avail` list */
static int place_items(env_t* e, ngo_mt* mt, int32_t* avail, int* n_avail, int item, int qty) {
    int ms = e->ms, count = 0;
    int agent = e->pose[0] * ms + e->pose[1];
    while (count != qty) {
        if (*n_avail < 1) return NGW_ERR_PLACEMENT;                   /* the reference asserts here */
        int idx = (int)ngo_randint(mt, 0, (uint32_t)*n_avail);
        int cell = avail[idx];
        if (cell != agent) {
            int r = cell / ms, c = cell % ms;
            if (CELL(e, r, c) == 0 && CELL(e, r - 1, c) == 0 && CELL(e, r + 1, c) == 0 && CELL(e, r, c - 1) == 0 &&
                CELL(e, r, c + 1) == 0) {
                CELL(e, r, c) = (int8_t)item;
                count++;
            }
        }
        memmove(&avail[idx], &avail[idx + 1], (size_t)(*n_avail - idx - 1) * sizeof(int32_t));   /* list.pop(idx) */
        (*n_avail)--;
    }
    return 0;
}

/* Runs ops [op_begin, op_end) of the reset program; do_base != 0 first runs the base reset.
 * Splitting lets the caller take the LidarInFront reset observation where the reference takes it. */
int ngo_reset_legacy(const ngw_config* cfg, int ms, ngo_mt* mt, int8_t* map, uint8_t* pose, int32_t* inv,
                     int do_base, int op_begin, int op_end) {
    env_t e = {cfg, ms, map, pose, inv};
    int n_cells = ms * ms, rc = 0;
    int32_t* cells = (int32_t*)malloc(sizeof(int32_t) * (size_t)n_cells);
    if (do_base) {                                                     /* pogostick_v1_env.py:118-157 */
        for (int i = 0; i < cfg->n_items; i++) inv[i] = 0;
        pose[3] = 0;
        for (int r = 0; r < ms; r++)
            for (int c = 0; c < ms; c++)
                CELL(&e, r, c) = (r == 0 || c == 0 || r == ms - 1 || c == ms - 1) ? (int8_t)cfg->id_wall : 0;
        int n_avail = 0;
        for (int r = 2; r < ms - 2; r++)
            for (int c = 2; c < ms - 2; c++) cells[n_avail++] = r * ms + c;
        int idx = (int)ngo_randint(mt, 0, (uint32_t)n_avail);          /* agent cell (stays in the list) */
        pose[0] = (uint8_t)(cells[idx] / ms); pose[1] = (uint8_t)(cells[idx] % ms);
        pose[2] = (uint8_t)ngo_randint(mt, 0, 4);                      /* choice(['NORTH','SOUTH','WEST','EAST']) */
        for (int i = 0; i < cfg->n_place && rc == 0; i++)
            rc = place_items(&e, mt, cells, &n_avail, cfg->place_item[i], cfg->place_qty[i]);
    }
    for (int k = op_begin; k < op_end && k < cfg->n_reset_ops && rc == 0; k++) {
        const ngw_reset_op* op = &cfg->reset_ops[k];
        if (op->kind == NGW_RESET_INVSET) { inv[op->a] = op->lo; continue; }
        if (op->kind == NGW_RESET_TREETAP) {                           /* pogostick_v0_env.py:155-178 */
            int n_logs = 0, agent = pose[0] * ms + pose[1];
            for (int i = 0; i < n_cells; i++) if (map[i] == op->b) cells[n_logs++] = i;   /* np.where, row-major */
            if (n_logs <= 1) { rc = NGW_ERR_PLACEMENT; break; }        /* assert len(result[0]) > 1 */
            for (;;) {
                int direction = (int)ngo_randint(mt, 0, 4);            /* np.random.choice(['NORTH','SOUTH','WEST','EAST']) */
                int log = cells[ngo_randint(mt, 0, (uint32_t)n_logs)]; /* np.random.choice(len(result[0])) */
                int r = log / ms, c = log % ms;
                int tr = r + (direction == NGW_SOUTH) - (direction == NGW_NORTH);
                int tc = c + (direction == NGW_EAST) - (direction == NGW_WEST);
                if (tr >= 0 && tr <= ms - 1 && tc >= 0 && tc <= ms - 1 && map[tr * ms + tc] == 0 && tr * ms + tc != agent) {
                    map[tr * ms + tc] = (int8_t)op->a;
                    break;                                             /* a tree_tap now exists */
                }
            }
            continue;
        }
        int n = 0;                                                     /* np.where(...) is row-major */
        for (int i = 0; i < n_cells; i++) {
            int id = map[i], take;
            if (op->kind == NGW_RESET_FENCE) take = (id != 0 && id != cfg->id_wall);
            else if (op->kind == NGW_RESET_ADDITEM) take = (id == 0);
            else take = (id == op->a);
            if (take) cells[n++] = i;
        }
        ngo_shuffle_i32(mt, cells, n);                                 /* shuffled indices == shuffled cells */
        int pct = (int)ngo_randint(mt, op->lo, op->hi);
        int m = percent_count(n, pct);
        int agent = pose[0] * ms + pose[1];
        for (int i = 0; i < m && i < n; i++) {
            int r = cells[i] / ms, c = cells[i] % ms;
            if (op->kind == NGW_RESET_FENCE) {                         /* add_fence_around, pogostick_v1_env.py:524-536 */
                for (int rr = r - 1; rr <= r + 1; rr++)
                    for (int cc = c - 1; cc <= c + 1; cc++)
                        if (CELL(&e, rr, cc) == 0 && rr * ms + cc != agent) CELL(&e, rr, cc) = (int8_t)op->a;
            } else if (cells[i] != agent) {
                CELL(&e, r, c) = (int8_t)(op->kind == NGW_RESET_ADDITEM ? op->a : op->b);
            }
        }
    }
    free(cells);
    return rc;
}

/* ------------------------------------------------------------------ batched, threaded driver (CPU baseline) */
typedef struct {
    const ngw_config* cfgs; const uint8_t* cfg_id; int ms; int64_t begin, end;
    int8_t* map; uint8_t* pose; int32_t* inv; int inv_stride;
    const int32_t* actions; int32_t* obs; int obs_stride;
    float* reward; uint8_t* done; float* cost; uint8_t* result; uint32_t* err; uint16_t* msg;
} job_t;

static void* batch_worker(void* arg) {
    job_t* j = (job_t*)arg;
    int cells = j->ms * j->ms;
    for (int64_t i = j->begin; i < j->end; i++) {
        const ngw_config* cfg = &j->cfgs[j->cfg_id ? j->cfg_id[i] : 0];
        int8_t* map = j->map + i * cells;
        uint8_t* pose = j->pose + i * 4;
        int32_t* inv = j->inv + i * j->inv_stride;
        int rc = ngo_step(cfg, j->ms, map, pose, inv, j->actions[i], &j->reward[i], &j->done[i], &j->cost[i],
                          &j->result[i], j->msg ? &j->msg[i] : NULL);
        if (j->err) j->err[i] |= (uint32_t)rc;
        if (j->obs) {
            int32_t* o = j->obs + i * j->obs_stride;
            int d = cfg->n_lidar_items * cfg->n_beams + cfg->n_inv_obs;
            ngo_observe(cfg, j->ms, map, pose, inv, o);
            for (int k = d; k < j->obs_stride; k++) o[k] = 0;
        }
    }
    return NULL;
}

/* One lock-step pass over n envs with n_threads host threads (envs are independent).  msg (uint16 [n]) may be NULL. */
int ngo_step_batch(const ngw_config* cfgs, const uint8_t* cfg_id, int ms, int64_t n, int8_t* map, uint8_t* pose,
                   int32_t* inv, int inv_stride, const int32_t* actions, int32_t* obs, int obs_stride, float* reward,
                   uint8_t* done, float* cost, uint8_t* result, uint32_t* err, int n_threads, uint16_t* msg) {
    if (n_threads < 1) n_threads = 1;
    if (n_threads > 1024) n_threads = 1024;
    job_t* jobs = (job_t*)malloc(sizeof(job_t) * (size_t)n_threads);
    pthread_t* th = (pthread_t*)malloc(sizeof(pthread_t) * (size_t)n_threads);
    int64_t per = (n + n_threads - 1) / n_threads;
    for (int t = 0; t < n_threads; t++) {
        int64_t b = t * per, e = b + per;
        if (b > n) b = n;
        if (e > n) e = n;
        job_t j = {cfgs, cfg_id, ms, b, e, map, pose, inv, inv_stride, actions, obs, obs_stride,
                   reward, done, cost, result, err, msg};
        jobs[t] = j;
        if (n_threads == 1) batch_worker(&jobs[t]);
        else pthread_create(&th[t], NULL, batch_worker, &jobs[t]);
    }
    if (n_threads > 1)
        for (int t = 0; t < n_threads; t++) pthread_join(th[t], NULL);
    free(jobs); free(th);
    return 0;
}

/* n_steps consecutive steps of every env, no lock-step barrier between threads (envs are independent): thread t
 * owns a contiguous slice and runs it through all steps; step s uses actions[(s % n_action_sets)][env].
 * This is the CPU-baseline driver: thread start-up is paid once per call, not once per step. */
typedef struct { job_t j; const int32_t* action_sets; int n_action_sets; int n_steps; int64_t n; } roll_t;

static void* rollout_worker(void* arg) {
    roll_t* r = (roll_t*)arg;
    for (int s = 0; s < r->n_steps; s++) {
        r->j.actions = r->action_sets + (int64_t)(s % r->n_action_sets) * r->n;
        batch_worker(&r->j);
    }
    return NULL;
}

int ngo_rollout(const ngw_config* cfgs, const uint8_t* cfg_id, int ms, int64_t n, int8_t* map, uint8_t* pose,
                int32_t* inv, int inv_stride, const int32_t* action_sets, int n_action_sets, int n_steps, int32_t* obs,
                int obs_stride, float* reward, uint8_t* done, float* cost, uint8_t* result, uint32_t* err,
                int n_threads) {
    if (n_threads < 1) n_threads = 1;
    if (n_threads > 1024) n_threads = 1024;
    roll_t* jobs = (roll_t*)malloc(sizeof(roll_t) * (size_t)n_threads);
    pthread_t* th = (pthread_t*)malloc(sizeof(pthread_t) * (size_t)n_threads);
    int64_t per = (n + n_threads - 1) / n_threads;
    for (int t = 0; t < n_threads; t++) {
        int64_t b = t * per, e = b + per;
        if (b > n) b = n;
        if (e > n) e = n;
        job_t j = {cfgs, cfg_id, ms, b, e, map, pose, inv, inv_stride, NULL, obs, obs_stride,
                   reward, done, cost, result, err, NULL};
        jobs[t].j = j; jobs[t].action_sets = action_sets; jobs[t].n_action_sets = n_action_sets;
        jobs[t].n_steps = n_steps; jobs[t].n = n;
        if (n_threads == 1) rollout_worker(&jobs[t]);
        else pthread_create(&th[t], NULL, rollout_worker, &jobs[t]);
    }
    if (n_threads > 1)
        for (int t = 0; t < n_threads; t++) pthread_join(th[t], NULL);
    free(jobs); free(th);
    return 0;
}

/* Legacy-stream resets of envs [0, n): env i is seeded with seed0 + i (np.random.seed) — how the parity
 * harness produces reference-exact reset states on a box where the reference itself is absent. */
int ngo_reset_batch(const ngw_config* cfgs, const uint8_t* cfg_id, int ms, int64_t n, uint32_t seed0, int8_t* map,
                    uint8_t* pose, int32_t* inv, int inv_stride, uint32_t* err) {
    int cells = ms * ms;
    for (int64_t i = 0; i < n; i++) {
        const ngw_config* cfg = &cfgs[cfg_id ? cfg_id[i] : 0];
        ngo_mt mt;
        ngo_mt_seed(&mt, seed0 + (uint32_t)i);
        int32_t* v = inv + i * inv_stride;
        for (int k = 0; k < inv_stride; k++) v[k] = 0;
        int rc = ngo_reset_legacy(cfg, ms, &mt, map + i * cells, pose + i * 4, v, 1, 0, cfg->n_reset_ops);
        if (err) err[i] = (uint32_t)rc;
    }
    return 0;
}

/* ==================================================================================================================
 * RESTATEMENT OF THE DEVICE'S GENERATOR (gym_novel_gridworlds_b200/csrc/ngw_device.cuh: Philox, RandomPolicy,
 * reset_env_warp).  Everything above restates the reference; this section does not.  The device's map generator has the
 * reference's DISTRIBUTION, not its stream, so it cannot be pinned by the golden traces: this is the CPU statement of its
 * contract, written from that contract (not from the warp code), against which tests/test_gpu_reset_exact.py compares
 * every GPU reset and random-policy draw bit for bit.
 *   Philox4x32-10: counter = (gid lo, gid hi, episode word, (stream << 20) | block), key = (seed lo, seed hi); next()
 *     returns words 0..3 of block 0, then of block 1, ...; below(n) = mask (0xFFFFFFFF >> clz(n - 1)) and reject.
 *   Base (stream 0): walls on the border, agent = below(side^2), facing = below(4), then each item copy takes up to
 *     8 side^2 draws for a placeable cell; failing that, below(good) picks among the placeable cells in row-major order.
 *   Op k (stream 1 + k): INVSET, TREETAP (4096 attempts over (direction, log)), and FENCE / ADDITEM / REPLACE, which pick
 *     the `take` candidates of smallest (key, cell index), key of cell i = word i % 4 of block 1 + i / 4 — except that a
 *     tie of more than 32 candidates on the boundary key goes by the device's arrival order (i >> 7, i & 3, i >> 2).
 *   Random policy: word t & 3 of block 0 at episode word t >> 2, stream 0xFFF; action = high half of x * n, Lemire's
 *     rejection continuing on stream 0xFFE at episode word t.
 * ================================================================================================================== */
void ngo_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
    uint32_t x0 = ctr[0], x1 = ctr[1], x2 = ctr[2], x3 = ctr[3], k0 = key[0], k1 = key[1];
    for (int r = 0; r < 10; r++) {
        uint64_t p0 = (uint64_t)0xD2511F53u * x0, p1 = (uint64_t)0xCD9E8D57u * x2;
        uint32_t y0 = (uint32_t)(p1 >> 32) ^ x1 ^ k0, y1 = (uint32_t)p1;
        uint32_t y2 = (uint32_t)(p0 >> 32) ^ x3 ^ k1, y3 = (uint32_t)p0;
        x0 = y0; x1 = y1; x2 = y2; x3 = y3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = x0; out[1] = x1; out[2] = x2; out[3] = x3;
}

typedef struct {
    uint32_t ctr[4], key[2], word[4];
    uint32_t block;    /* next block to generate */
    int used;          /* words of `word` already returned (4: generate the next block first) */
} ngo_pstream;

static void ps_block(uint64_t seed, uint64_t gid, uint32_t episode, uint32_t stream, uint32_t block, uint32_t out[4]) {
    uint32_t ctr[4] = {(uint32_t)gid, (uint32_t)(gid >> 32), episode, (stream << 20) | block};
    uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
    ngo_philox4x32_10(ctr, key, out);
}

static void ps_init(ngo_pstream* s, uint64_t seed, uint64_t gid, uint32_t episode, uint32_t stream) {
    s->ctr[0] = (uint32_t)gid; s->ctr[1] = (uint32_t)(gid >> 32); s->ctr[2] = episode; s->ctr[3] = stream << 20;
    s->key[0] = (uint32_t)seed; s->key[1] = (uint32_t)(seed >> 32);
    s->block = 0; s->used = 4;
}

static uint32_t ps_next(ngo_pstream* s) {
    if (s->used == 4) {
        uint32_t ctr[4] = {s->ctr[0], s->ctr[1], s->ctr[2], s->ctr[3] | s->block};
        ngo_philox4x32_10(ctr, s->key, s->word);
        s->block++; s->used = 0;
    }
    return s->word[s->used++];
}

static uint32_t ps_below(ngo_pstream* s, uint32_t n) {
    uint32_t max = n - 1u, mask = max;
    if (max == 0) return 0;
    mask |= mask >> 1; mask |= mask >> 2; mask |= mask >> 4; mask |= mask >> 8; mask |= mask >> 16;
    uint32_t v;
    do { v = ps_next(s) & mask; } while (v > max);
    return v;
}

/* the first `count` outputs of below(n) on one stream (the test of the word stream and of the rejection rate) */
void ngo_philox_below(uint64_t seed, uint64_t gid, uint32_t episode, uint32_t stream, uint32_t n, int64_t count,
                      uint32_t* out, uint32_t* words_used) {
    ngo_pstream s;
    ps_init(&s, seed, gid, episode, stream);
    for (int64_t i = 0; i < count; i++) out[i] = ps_below(&s, n);
    if (words_used) *words_used = s.block * 4u - (uint32_t)(4 - s.used);
}

/* The random policy's action for step t of env gid (config with n actions); *branch = 0: plain draw, 1: the low half
 * was below n and the draw was kept, 2: it was below (2^32 - n) mod n and continued on stream 0xFFE. */
int32_t ngo_policy_draw(uint64_t seed, uint64_t gid, uint32_t t, uint32_t n, int* branch) {
    uint32_t w[4];
    ps_block(seed, gid, t >> 2, 0xFFF, 0, w);
    uint64_t m = (uint64_t)w[t & 3u] * n;
    int br = 0;
    if ((uint32_t)m < n) {
        uint32_t thr = (0u - n) % n;
        br = (uint32_t)m < thr ? 2 : 1;
        ngo_pstream s;
        ps_init(&s, seed, gid, t, 0xFFE);
        while ((uint32_t)m < thr) m = (uint64_t)ps_next(&s) * n;
    }
    if (branch) *branch = br;
    return (int32_t)(m >> 32);
}

/* What a reset did, summed over envs: the events the exact tests must see happen. */
enum {
    NGO_RS_FALLBACK = 0,      /* item copies placed by the enumeration after 8 side^2 failed draws */
    NGO_RS_PLACE_FAIL,        /* base placements that found no placeable cell (PLACEMENT, remaining items skipped) */
    NGO_RS_TREETAP_FAIL,      /* TREETAP ops that flagged PLACEMENT */
    NGO_RS_SUBSET,            /* FENCE / ADDITEM / REPLACE ops with 0 < take */
    NGO_RS_ALL_WIN,           /* ... whose boundary bin won whole (take == n, or a radix bin boundary) */
    NGO_RS_LIST,              /* ... decided by ranking a boundary list of <= 32 candidates by (key, cell) */
    NGO_RS_ARRIVAL,           /* ... where > 32 candidates tied on the boundary key and arrival order decided */
    NGO_RS_COUNT = 8
};

typedef struct { uint32_t key; int32_t cell; } ngo_cand;

static int cand_by_key_cell(const void* a, const void* b) {
    const ngo_cand *x = (const ngo_cand*)a, *y = (const ngo_cand*)b;
    if (x->key != y->key) return x->key < y->key ? -1 : 1;
    return x->cell < y->cell ? -1 : x->cell > y->cell;
}

static int64_t arrival_rank(int32_t i) { return ((int64_t)(i >> 7) << 40) | ((int64_t)(i & 3) << 32) | (i >> 2); }

static int cand_by_arrival(const void* a, const void* b) {
    int64_t x = arrival_rank(((const ngo_cand*)a)->cell), y = arrival_rank(((const ngo_cand*)b)->cell);
    return x < y ? -1 : x > y;
}

static int placeable_at(const int8_t* m, int ms, int r, int c) {
    const int8_t* p = m + r * ms + c;
    return p[0] == 0 && p[-ms] == 0 && p[ms] == 0 && p[-1] == 0 && p[1] == 0;
}

/* The outcome of the device's radix-select for `take` of the n candidates sorted by (key, cell): 0 = the boundary bin
 * wins whole, 1 = a boundary list of <= 32 is ranked, 2 = more than 32 identical boundary keys, arrival order.  Bins are
 * the top 8, 16, 24, 32 key bits of the take-th smallest key; the select narrows while fewer than all of the bin's
 * candidates are still needed and the bin holds more than 32. */
static int radix_outcome(const ngo_cand* c, int n, int take) {
    const uint32_t kth = c[take - 1].key;
    int bits = 0, remaining = take, bin_count = n;
    while (remaining < bin_count && bin_count > 32 && bits < 32) {
        bits += 8;
        int less = 0, same = 0;
        for (int i = 0; i < n; i++) {
            uint32_t top = c[i].key >> (32 - bits), want = kth >> (32 - bits);
            less += top < want; same += top == want;
        }
        remaining = take - less;
        bin_count = same;
    }
    if (remaining >= bin_count) return 0;
    return (bits >= 32 && bin_count > 32) ? 2 : 1;
}

/* Ops [op_begin, op_end) of the reset program, do_base != 0 running the base first, at (seed, gid, episode word).
 * Returns the PLACEMENT flag of what ran; counters (NGO_RS_COUNT) may be NULL. */
int ngo_reset_philox(const ngw_config* cfg, int ms, uint64_t seed, uint64_t gid, uint32_t episode, uint32_t key_mask,
                     int8_t* map, uint8_t* pose, int32_t* inv, int inv_stride, int do_base, int op_begin, int op_end,
                     int64_t* counters) {
    const int cells = ms * ms, wall = cfg->id_wall;
    int64_t dummy[NGO_RS_COUNT];
    int64_t* ct = counters ? counters : dummy;
    int err = 0;
    if (do_base) {
        for (int i = 0; i < inv_stride; i++) inv[i] = 0;
        pose[3] = 0;
        for (int r = 0; r < ms; r++)
            for (int c = 0; c < ms; c++) map[r * ms + c] = (r == 0 || c == 0 || r == ms - 1 || c == ms - 1) ? (int8_t)wall : 0;
        ngo_pstream s;
        ps_init(&s, seed, gid, episode, 0);
        const int side = ms - 4;
        const uint32_t n_av = (uint32_t)(side * side);
        uint32_t a = ps_below(&s, n_av);
        pose[0] = (uint8_t)(2 + a / side); pose[1] = (uint8_t)(2 + a % side);
        pose[2] = (uint8_t)ps_below(&s, 4);
        const int agent = pose[0] * ms + pose[1];
        int stop = 0;
        for (int i = 0; i < cfg->n_place && !stop; i++) {
            for (int count = 0; count < cfg->place_qty[i]; count++) {
                int where = -1;
                for (uint32_t attempt = 0; attempt < 8 * n_av && where < 0; attempt++) {
                    uint32_t d = ps_below(&s, n_av);
                    int r = 2 + (int)(d / side), c = 2 + (int)(d % side);
                    if (r * ms + c != agent && placeable_at(map, ms, r, c)) where = r * ms + c;
                }
                if (where < 0) {
                    uint32_t good = 0;
                    for (int r = 2; r <= ms - 3; r++)
                        for (int c = 2; c <= ms - 3; c++) good += r * ms + c != agent && placeable_at(map, ms, r, c);
                    if (good == 0) { err |= NGW_ERR_PLACEMENT; ct[NGO_RS_PLACE_FAIL]++; stop = 1; break; }
                    uint32_t pick = ps_below(&s, good);
                    for (int r = 2; r <= ms - 3 && where < 0; r++)
                        for (int c = 2; c <= ms - 3 && where < 0; c++)
                            if (r * ms + c != agent && placeable_at(map, ms, r, c) && pick-- == 0) where = r * ms + c;
                    ct[NGO_RS_FALLBACK]++;
                }
                map[where] = (int8_t)cfg->place_item[i];
            }
        }
    }
    const int agent = pose[0] * ms + pose[1];
    if (op_end > cfg->n_reset_ops) op_end = cfg->n_reset_ops;
    ngo_cand* cand = (ngo_cand*)malloc(sizeof(ngo_cand) * (size_t)cells);
    for (int k = op_begin; k < op_end; k++) {
        const ngw_reset_op* op = &cfg->reset_ops[k];
        const uint32_t stream = 1u + (uint32_t)k;
        if (op->kind == NGW_RESET_INVSET) { inv[op->a] = op->lo; continue; }
        if (op->kind == NGW_RESET_TREETAP) {
            int n_logs = 0, target = -1;
            for (int i = 0; i < cells; i++) n_logs += map[i] == (int8_t)op->b;
            if (n_logs > 1) {
                ngo_pstream s;
                ps_init(&s, seed, gid, episode, stream);
                for (int attempt = 0; attempt < 4096 && target < 0; attempt++) {
                    int direction = (int)ps_below(&s, 4);
                    int which = (int)ps_below(&s, (uint32_t)n_logs), log = -1;
                    for (int i = 0; i < cells && log < 0; i++)
                        if (map[i] == (int8_t)op->b && which-- == 0) log = i;
                    int r = log / ms, c = log % ms;
                    int tr = r + (direction == NGW_SOUTH) - (direction == NGW_NORTH);
                    int tc = c + (direction == NGW_EAST) - (direction == NGW_WEST);
                    if (tr >= 0 && tr < ms && tc >= 0 && tc < ms && map[tr * ms + tc] == 0 && tr * ms + tc != agent)
                        target = tr * ms + tc;
                }
            }
            if (target < 0) { err |= NGW_ERR_PLACEMENT; ct[NGO_RS_TREETAP_FAIL]++; continue; }
            map[target] = (int8_t)op->a;
            continue;
        }
        int n = 0;
        for (int i = 0; i < cells; i++) {
            int id = map[i];
            int is = op->kind == NGW_RESET_FENCE ? (id != 0 && id != wall) : op->kind == NGW_RESET_ADDITEM ? id == 0 : id == op->a;
            if (!is) continue;
            uint32_t w[4];
            ps_block(seed, gid, episode, stream, 1u + (uint32_t)(i / 4), w);
            cand[n].key = w[i % 4] & key_mask;
            cand[n].cell = i;
            n++;
        }
        ngo_pstream s;
        ps_init(&s, seed, gid, episode, stream);
        const int pct = op->lo + (int)ps_below(&s, (uint32_t)(op->hi - op->lo));
        int take = percent_count(n, pct);
        if (take > n) take = n;
        if (take <= 0) continue;
        ct[NGO_RS_SUBSET]++;
        qsort(cand, (size_t)n, sizeof(ngo_cand), cand_by_key_cell);
        const int outcome = radix_outcome(cand, n, take);
        ct[outcome == 0 ? NGO_RS_ALL_WIN : outcome == 1 ? NGO_RS_LIST : NGO_RS_ARRIVAL]++;
        if (outcome == 2) {                                /* the tied group [lo, hi) is re-ordered by arrival */
            int lo = take - 1, hi = take;
            while (lo > 0 && cand[lo - 1].key == cand[take - 1].key) lo--;
            while (hi < n && cand[hi].key == cand[take - 1].key) hi++;
            qsort(cand + lo, (size_t)(hi - lo), sizeof(ngo_cand), cand_by_arrival);
        }
        for (int j = 0; j < take; j++) {
            const int i = cand[j].cell;
            if (op->kind == NGW_RESET_FENCE) {             /* add_fence_around the winner (fences only go into air) */
                int r = i / ms, c = i % ms;
                for (int rr = r - 1; rr <= r + 1; rr++)
                    for (int cc = c - 1; cc <= c + 1; cc++)
                        if (rr >= 0 && rr < ms && cc >= 0 && cc < ms && map[rr * ms + cc] == 0 && rr * ms + cc != agent)
                            map[rr * ms + cc] = (int8_t)op->a;
            } else if (i != agent) {
                map[i] = (int8_t)(op->kind == NGW_RESET_ADDITEM ? op->a : op->b);
            }
        }
    }
    free(cand);
    return err;
}

/* Device-generator resets of envs [0, n) with n_threads host threads: env i (skipped where mask[i] == 0) is reset at
 * gid first_gid + i and episode word episode[i]; its observation (obs may be NULL) is taken after k_obs[i] ops (NULL:
 * the config's reset_obs_after_ops).  err[i] is assigned the PLACEMENT flag; counters [NGO_RS_COUNT] are summed. */
typedef struct {
    const ngw_config* cfgs; const uint8_t* cfg_id; int ms; int64_t begin, end;
    uint64_t seed, first_gid; const uint32_t* episode; uint32_t key_mask; const uint8_t* mask; const int32_t* k_obs;
    int8_t* map; uint8_t* pose; int32_t* inv; int inv_stride; int32_t* obs; int obs_stride; uint32_t* err;
    int64_t counters[NGO_RS_COUNT];
} preset_t;

static void* preset_worker(void* arg) {
    preset_t* j = (preset_t*)arg;
    const int cells = j->ms * j->ms;
    for (int64_t i = j->begin; i < j->end; i++) {
        if (j->mask && !j->mask[i]) continue;
        const ngw_config* cfg = &j->cfgs[j->cfg_id ? j->cfg_id[i] : 0];
        int8_t* map = j->map + i * cells;
        uint8_t* pose = j->pose + i * 4;
        int32_t* inv = j->inv + i * j->inv_stride;
        const uint64_t gid = j->first_gid + (uint64_t)i;
        int k = j->k_obs ? j->k_obs[i] : cfg->reset_obs_after_ops;
        int rc = ngo_reset_philox(cfg, j->ms, j->seed, gid, j->episode[i], j->key_mask, map, pose, inv, j->inv_stride, 1, 0,
                                  k, j->counters);
        if (j->obs) {
            int32_t* o = j->obs + i * j->obs_stride;
            for (int q = 0; q < j->obs_stride; q++) o[q] = 0;
            if (cfg->n_beams > 0) ngo_observe(cfg, j->ms, map, pose, inv, o);
        }
        rc |= ngo_reset_philox(cfg, j->ms, j->seed, gid, j->episode[i], j->key_mask, map, pose, inv, j->inv_stride, 0, k,
                               NGW_MAX_RESET_OPS, j->counters);
        if (j->err) j->err[i] = (uint32_t)rc;
    }
    return NULL;
}

int ngo_reset_philox_batch(const ngw_config* cfgs, const uint8_t* cfg_id, int ms, int64_t n, uint64_t seed,
                           uint64_t first_gid, const uint32_t* episode, uint32_t key_mask, const uint8_t* mask,
                           const int32_t* k_obs, int8_t* map, uint8_t* pose, int32_t* inv, int inv_stride, int32_t* obs,
                           int obs_stride, uint32_t* err, int64_t* counters, int n_threads) {
    if (n_threads < 1) n_threads = 1;
    if (n_threads > 1024) n_threads = 1024;
    preset_t* jobs = (preset_t*)calloc((size_t)n_threads, sizeof(preset_t));
    pthread_t* th = (pthread_t*)malloc(sizeof(pthread_t) * (size_t)n_threads);
    int64_t per = (n + n_threads - 1) / n_threads;
    for (int t = 0; t < n_threads; t++) {
        int64_t b = t * per, e = b + per;
        if (b > n) b = n;
        if (e > n) e = n;
        preset_t j = {cfgs, cfg_id, ms, b, e, seed, first_gid, episode, key_mask, mask, k_obs, map, pose, inv, inv_stride,
                      obs, obs_stride, err, {0}};
        jobs[t] = j;
        if (n_threads == 1) preset_worker(&jobs[t]);
        else pthread_create(&th[t], NULL, preset_worker, &jobs[t]);
    }
    if (n_threads > 1)
        for (int t = 0; t < n_threads; t++) pthread_join(th[t], NULL);
    if (counters)
        for (int t = 0; t < n_threads; t++)
            for (int c = 0; c < NGO_RS_COUNT; c++) counters[c] += jobs[t].counters[c];
    free(jobs); free(th);
    return 0;
}

/* out[s][i] = ngo_policy_draw(seed, first_gid + i, t0 + s, n_actions[i]) for s < n_steps, i < n; branch (may be NULL)
 * receives the branch taken, laid out like out. */
typedef struct {
    uint64_t seed, first_gid; int64_t n, begin, end; const int32_t* n_actions; uint32_t t0; int n_steps;
    int32_t* out; uint8_t* branch;
} pdraw_t;

static void* pdraw_worker(void* arg) {
    pdraw_t* j = (pdraw_t*)arg;
    for (int s = 0; s < j->n_steps; s++)
        for (int64_t i = j->begin; i < j->end; i++) {
            int br;
            j->out[s * j->n + i] = ngo_policy_draw(j->seed, j->first_gid + (uint64_t)i, j->t0 + (uint32_t)s,
                                                   (uint32_t)j->n_actions[i], &br);
            if (j->branch) j->branch[s * j->n + i] = (uint8_t)br;
        }
    return NULL;
}

int ngo_policy_draw_batch(uint64_t seed, uint64_t first_gid, int64_t n, const int32_t* n_actions, uint32_t t0, int n_steps,
                          int32_t* out, uint8_t* branch, int n_threads) {
    if (n_threads < 1) n_threads = 1;
    if (n_threads > 1024) n_threads = 1024;
    pdraw_t* jobs = (pdraw_t*)malloc(sizeof(pdraw_t) * (size_t)n_threads);
    pthread_t* th = (pthread_t*)malloc(sizeof(pthread_t) * (size_t)n_threads);
    int64_t per = (n + n_threads - 1) / n_threads;
    for (int t = 0; t < n_threads; t++) {
        int64_t b = t * per, e = b + per;
        if (b > n) b = n;
        if (e > n) e = n;
        pdraw_t j = {seed, first_gid, n, b, e, n_actions, t0, n_steps, out, branch};
        jobs[t] = j;
        if (n_threads == 1) pdraw_worker(&jobs[t]);
        else pthread_create(&th[t], NULL, pdraw_worker, &jobs[t]);
    }
    if (n_threads > 1)
        for (int t = 0; t < n_threads; t++) pthread_join(th[t], NULL);
    free(jobs); free(th);
    return 0;
}

int ngo_sizeof_config(void) { return (int)sizeof(ngw_config); }
int ngo_sizeof_mt(void) { return (int)sizeof(ngo_mt); }
