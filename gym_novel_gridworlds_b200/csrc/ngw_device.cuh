// ngw_device.cuh — per-env device code of the batched NovelGridworld simulator (sm_100a).
//
// One lane owns one environment.  The lane's grid row, inventory row and observation row live in
// shared memory (staged by the kernels in ngw_step.cuh); everything here works on those rows through
// plain pointers, so the same code also runs straight on global memory in the (cold) reset kernel.
//
// Semantics follow the reference file:line cited at each function (paths under
// /root/reference/gym_novel_gridworlds/); the wrapper chain arrives flattened as an ngw_config.
#pragma once
#include <stdint.h>
#include "../../include/ngw.h"

namespace ngw {

// ------------------------------------------------------------------ Philox4x32-10 (counter-based RNG)
// counter = (global env id lo, hi, episode index, (stream << 20) | block), key = seed: draws depend only on
// (seed, global env id, episode, stream, position) => identical episodes for any sharding over GPUs.
struct Philox {
    uint32_t c0, c1, c2, c3base, k0, k1;
    uint32_t buf[4];
    uint32_t blk;
    int have;

    __device__ __forceinline__ void init(uint64_t seed, uint64_t gid, uint32_t episode, uint32_t stream) {
        c0 = (uint32_t)gid; c1 = (uint32_t)(gid >> 32); c2 = episode; c3base = stream << 20;
        k0 = (uint32_t)seed; k1 = (uint32_t)(seed >> 32);
        blk = 0; have = 0;
    }
    __device__ __forceinline__ void refill() {
        uint32_t x0 = c0, x1 = c1, x2 = c2, x3 = c3base | blk, a = k0, b = k1;
#pragma unroll
        for (int r = 0; r < 10; r++) {
            uint32_t hi0 = __umulhi(0xD2511F53u, x0), lo0 = 0xD2511F53u * x0;
            uint32_t hi1 = __umulhi(0xCD9E8D57u, x2), lo1 = 0xCD9E8D57u * x2;
            uint32_t y0 = hi1 ^ x1 ^ a, y1 = lo1, y2 = hi0 ^ x3 ^ b, y3 = lo0;
            x0 = y0; x1 = y1; x2 = y2; x3 = y3;
            a += 0x9E3779B9u; b += 0xBB67AE85u;
        }
        buf[0] = x0; buf[1] = x1; buf[2] = x2; buf[3] = x3;
        blk++; have = 4;
    }
    __device__ __forceinline__ uint32_t next() {
        if (have == 0) refill();
        have--;
        // static indexing keeps buf in registers
        return have == 3 ? buf[0] : have == 2 ? buf[1] : have == 1 ? buf[2] : buf[3];
    }
    // unbiased uniform integer in [0, n), n >= 1 (mask + rejection, like NumPy's legacy bounded draw)
    __device__ __forceinline__ uint32_t below(uint32_t n) {
        uint32_t max = n - 1;
        if (max == 0) return 0;
        uint32_t mask = 0xFFFFFFFFu >> __clz(max);
        uint32_t v;
        do { v = next() & mask; } while (v > max);
        return v;
    }
};

// On-device uniform random policy of the rollout kernels: one Philox block (counter = step / 4, stream 0xFFF) yields the
// draws of four consecutive steps; a draw becomes an action id in [0, n) by multiply-shift with Lemire's rejection (exact
// uniformity; a rejection — probability n / 2^32 — continues on stream 0xFFE of that step).
struct RandomPolicy {
    uint32_t w[4];
    __device__ __forceinline__ int draw(uint64_t seed, uint64_t gid, uint32_t t, uint32_t n) {
        if ((t & 3u) == 0u || t == first) {
            Philox pr;
            pr.init(seed, gid, t >> 2, 0xFFF);
            pr.refill();
            w[0] = pr.buf[0]; w[1] = pr.buf[1]; w[2] = pr.buf[2]; w[3] = pr.buf[3];
        }
        const uint32_t k = t & 3u;
        uint32_t x = k == 0 ? w[0] : k == 1 ? w[1] : k == 2 ? w[2] : w[3];
        uint64_t m = (uint64_t)x * n;
        if ((uint32_t)m < n) {                                        // rare: exact rejection threshold
            const uint32_t thr = (0u - n) % n;
            Philox pr;
            pr.init(seed, gid, t, 0xFFE);
            while ((uint32_t)m < thr) { x = pr.next(); m = (uint64_t)x * n; }
        }
        return (int)(m >> 32);
    }
    uint32_t first;                                                   // first step of this launch (its block must be generated)
};

// ------------------------------------------------------------------ per-env view
struct EnvRow {
    int8_t* m;                            // staged grid row [cells]
    int8_t* gm;                           // the same row in global memory (write-through of the few changed cells), or nullptr
    int32_t* inv;                         // staged inventory row
    int ms;
    int r, c, facing, sel;
    bool inv_dirty = false;               // the step changed the inventory row (inv_add): step1w_kernel stores only such rows
    __device__ __forceinline__ void set_pose(uchar4 ps) { r = ps.x; c = ps.y; facing = ps.z; sel = ps.w; }
    __device__ __forceinline__ uchar4 pose() const {
        return make_uchar4((unsigned char)r, (unsigned char)c, (unsigned char)facing, (unsigned char)sel);
    }
};

struct StepOut {
    int reward;
    int done;
    int result;
    float cost;
    int msg;        // enum ngw_msg | argument << 5
    int goal;       // the goal item is in the inventory after the step (done by success, not by fire / truncation)
    __device__ __forceinline__ void clear() { reward = 0; done = 0; result = 0; cost = 0.0f; msg = 0; goal = 0; }
};

// every inventory change a step makes goes through here (resets store whole rows and do not)
__device__ __forceinline__ void inv_add(EnvRow& e, int item, int delta) {
    e.inv[item] += delta;
    e.inv_dirty = true;
}

__device__ __forceinline__ int msg_of(int code, int arg) { return code | (arg << 5); }

__device__ __forceinline__ int cell(const EnvRow& e, int r, int c) { return e.m[r * e.ms + c]; }

__device__ __forceinline__ void set_cell(EnvRow& e, int r, int c, int v) {
    int idx = r * e.ms + c;
    e.m[idx] = (int8_t)v;
    if (e.gm) e.gm[idx] = (int8_t)v;
}

__device__ __forceinline__ bool in_mask(uint32_t mask, int item) { return (mask >> (item & 31)) & 1u; }

// update_block_in_front (pogostick_v1_env.py:369-383)
__device__ __forceinline__ void front_of(const EnvRow& e, int& fr, int& fc) {
    fr = e.r + (e.facing == NGW_SOUTH) - (e.facing == NGW_NORTH);
    fc = e.c + (e.facing == NGW_EAST) - (e.facing == NGW_WEST);
}

// bounds-checked neighbour test shared by is_block_in_front_next_to (pogostick_v1_env.py:391-411)
// and the fire_wall check (novelty_wrappers.py:1171-1184)
__device__ __forceinline__ bool next_to(const EnvRow& e, int r, int c, int item) {
    int hi = e.ms - 1;
    bool hit = false;
    if (r - 1 >= 0 && r - 1 <= hi && c >= 0 && c <= hi) hit |= cell(e, r - 1, c) == item;
    if (r + 1 >= 0 && r + 1 <= hi && c >= 0 && c <= hi) hit |= cell(e, r + 1, c) == item;
    if (c - 1 >= 0 && c - 1 <= hi && r >= 0 && r <= hi) hit |= cell(e, r, c - 1) == item;
    if (c + 1 >= 0 && c + 1 <= hi && r >= 0 && r <= hi) hit |= cell(e, r, c + 1) == item;
    return hit;
}

// grab_entities (pogostick_v1_env.py:538-554); the agent is always interior so the 3x3 is in bounds
__device__ __forceinline__ void grab_entities(EnvRow& e, const ngw_config& cfg) {
    uint32_t mask = cfg.entity_mask;
    if (mask == 0) return;
    for (int rr = e.r - 1; rr <= e.r + 1; rr++)
        for (int cc = e.c - 1; cc <= e.c + 1; cc++) {
            int id = cell(e, rr, cc);
            if (id != 0 && in_mask(mask, id)) {
                set_cell(e, rr, cc, 0);
                inv_add(e, id, 1);
            }
        }
}

// craft (pogostick_v1_env.py:413-474, bow_v1_env.py:386-441, novelty_wrappers.py:371-436)
__device__ __forceinline__ void craft(EnvRow& e, const ngw_config& cfg, int slot, StepOut& o) {
    const ngw_recipe& rc = cfg.recipes[slot];
    int missing = 0;
    int n_in = rc.n_inputs;
    for (int i = 0; i < n_in; i++) {
        int item = rc.in_item[i];
        bool have = (item != NGW_NONE) && (e.inv[item == NGW_NONE ? 0 : item] >= (int)rc.in_qty[i]);
        missing |= have ? 0 : (1 << i);
    }
    if (missing) {
        o.result = 0; o.cost = rc.cost_missing;
        o.msg = msg_of(NGW_MSG_MISSING, slot | (missing << 3));
        return;
    }
    if (rc.needs_table) {
        int fr, fc;
        front_of(e, fr, fc);
        if (cell(e, fr, fc) != cfg.id_crafting_table) {
            o.result = 0; o.cost = rc.cost_no_table; o.msg = NGW_MSG_NEED_TABLE;
            return;
        }
    }
    o.reward = rc.reward_ok;
    o.msg = msg_of(NGW_MSG_CRAFTED, rc.out_item);
    for (int i = 0; i < n_in; i++) inv_add(e, rc.in_item[i], -(int)rc.in_qty[i]);
    inv_add(e, rc.out_item, (int)rc.out_qty);
    o.cost = rc.cost_ok;
}

// terminal opcode: the innermost step body that finally handles the action, WITHOUT its trailing
// grab_entities / done block (applied by the caller, once, as the reference's paths all do)
__device__ __forceinline__ void terminal_op(EnvRow& e, const ngw_config& cfg, const ngw_action_entry a, StepOut& o) {
    int fr, fc;
    front_of(e, fr, fc);
    o.reward = -1; o.result = 1; o.cost = 0.0f; o.done = 0; o.msg = 0;   // pogostick_v1_env.py:239-242
    switch (a.op) {
        case NGW_OP_FORWARD:                                          // pogostick_v1_env.py:244-257
            if (cell(e, fr, fc) == 0) { e.r = fr; e.c = fc; } else { o.result = 0; o.msg = NGW_MSG_BLOCK_IN_PATH; }
            o.cost = 27.906975f;
            break;
        case NGW_OP_LEFT:                                             // N->W S->E W->S E->N  (0->2 1->3 2->1 3->0)
            e.facing = (0x0132 >> (e.facing * 4)) & 0xF; o.cost = 24.0f;
            break;
        case NGW_OP_RIGHT:                                            // N->E S->W W->N E->S  (0->3 1->2 2->0 3->1)
            e.facing = (0x1023 >> (e.facing * 4)) & 0xF; o.cost = 24.0f;
            break;
        case NGW_OP_BREAK: {
            int front = cell(e, fr, fc);
            o.cost = 3600.0f;
            if (in_mask(cfg.unbreakable_mask, front)) { o.result = 0; o.msg = msg_of(NGW_MSG_CANNOT_BREAK, front); break; }
            int variant = a.variant;
            if (variant == NGW_BRK_BASE) {                            // pogostick_v1_env.py:283-289
                set_cell(e, fr, fc, 0);
                inv_add(e, front, 1);
                if (in_mask(cfg.break_reward_mask, front)) o.reward = cfg.reward_intermediate;
            } else if (variant == NGW_BRK_INCREASE) {                 // novelty_wrappers.py:1444-1454
                set_cell(e, fr, fc, 0);
                inv_add(e, front, (a.arg == NGW_NONE || a.arg == front) ? 2 : 1);
                o.reward = cfg.reward_intermediate;
            } else {                                                  // axe / axetobreak, novelty_wrappers.py:55-81, 482-501
                bool has_axe = e.inv[a.arg] >= 1;
                bool wooden = has_axe && cfg.id_wooden_axe != NGW_NONE && e.sel == cfg.id_wooden_axe;
                bool iron = has_axe && !wooden && cfg.id_iron_axe != NGW_NONE && e.sel == cfg.id_iron_axe;
                if (wooden || iron) {
                    set_cell(e, fr, fc, 0);
                    inv_add(e, front, (variant == NGW_BRK_AXE_INC) ? 2 : 1);
                    o.reward = cfg.reward_intermediate;
                    o.cost = wooden ? 1800.0f : 900.0f;
                } else if (variant == NGW_BRK_AXETOBREAK) {
                    o.result = 0; o.msg = msg_of(NGW_MSG_NEED_AXE, a.arg);
                } else {                                              // breaks, but no reward even for tree_log (Q4)
                    set_cell(e, fr, fc, 0);
                    inv_add(e, front, 1);
                }
            }
            break;
        }
        case NGW_OP_PLACE_TREE_TAP:                                   // pogostick_v1_env.py:295-314
            o.cost = 300.0f;
            if (e.inv[cfg.id_tree_tap] >= 1 && cell(e, fr, fc) == 0) {
                set_cell(e, fr, fc, cfg.id_tree_tap);
                inv_add(e, cfg.id_tree_tap, -1);
                o.msg = NGW_MSG_TAP_PLACED;
                if (next_to(e, fr, fc, cfg.id_tree_log)) o.reward = cfg.reward_intermediate;
            } else {
                o.result = 0;
                o.msg = e.inv[cfg.id_tree_tap] >= 1 ? msg_of(NGW_MSG_BLOCK_EXISTS, cell(e, fr, fc)) : NGW_MSG_NOT_IN_INVENTORY;
            }
            break;
        case NGW_OP_EXTRACT_RUBBER:                                   // pogostick_v1_env.py:315-331, novelty_wrappers.py:1537-1551
            o.cost = 120.0f;
            if (cell(e, fr, fc) == cfg.id_tree_tap && next_to(e, fr, fc, cfg.id_tree_log)) {
                inv_add(e, cfg.id_rubber, a.arg);
                o.reward = cfg.reward_intermediate; o.cost = 50000.0f;
            } else {
                o.result = 0;
                o.msg = cell(e, fr, fc) == cfg.id_tree_tap ? NGW_MSG_NO_LOG_NEAR_TAP : NGW_MSG_NO_TAP;
            }
            break;
        case NGW_OP_EXTRACT_STRING:                                   // bow_v1_env.py:293-304, novelty_wrappers.py:1524-1536
            o.cost = 120.0f;
            if (cell(e, fr, fc) == cfg.id_wool) {
                inv_add(e, cfg.id_string, a.arg);
                set_cell(e, fr, fc, 0);
                o.reward = cfg.reward_intermediate; o.cost = 5000.0f;
            } else { o.result = 0; o.msg = NGW_MSG_NO_WOOL; }
            break;
        case NGW_OP_CRAFT:
            craft(e, cfg, a.arg, o);
            break;
        case NGW_OP_SELECT:                                           // pogostick_v1_env.py:338-347
            o.cost = 120.0f;
            if (a.arg != NGW_NONE && e.inv[a.arg] >= 1) e.sel = a.arg; else { o.result = 0; o.msg = NGW_MSG_NOT_IN_INVENTORY; }
            break;
        case NGW_OP_CHOP: {                                           // novelty_wrappers.py:1291-1307
            int front = cell(e, fr, fc);
            o.cost = 3600.0f * 1.2f;
            if (!in_mask(cfg.unbreakable_mask, front)) {
                set_cell(e, fr, fc, 0);
                inv_add(e, front, 2);
                o.reward = cfg.reward_intermediate;
            } else { o.result = 0; o.msg = msg_of(NGW_MSG_CANNOT_CHOP, front); }
            break;
        }
        case NGW_OP_JUMP: {                                           // novelty_wrappers.py:1363-1382
            int tr = e.r + 2 * (fr - e.r), tc = e.c + 2 * (fc - e.c);
            if (tr >= 0 && tr <= e.ms - 1 && tc >= 0 && tc <= e.ms - 1 && cell(e, tr, tc) == 0) { e.r = tr; e.c = tc; }
            else { o.result = 0; o.msg = NGW_MSG_BLOCK_IN_PATH; }
            o.cost = 27.906975f * 2.0f;
            break;
        }
        default: break;                                               // NGW_OP_NOOP
    }
}

// "Update after each step" (pogostick_v1_env.py:349-357 and its copies in every intercepting novelty)
__device__ __forceinline__ void post_step(EnvRow& e, const ngw_config& cfg, StepOut& o) {
    grab_entities(e, cfg);
    o.done = 0; o.goal = 0;
    if (e.inv[cfg.id_goal] >= 1) { o.reward = cfg.reward_done; o.done = 1; o.goal = 1; }
}

// One full reference step() through the flattened wrapper chain.  Layers are walked outermost-first
// (what each wrapper does before calling self.env.step), the terminal opcode runs if every
// FenceRestriction on the way let it through, then the layers' post blocks run innermost-first.
__device__ __forceinline__ void step_env(EnvRow& e, const ngw_config& cfg, const ngw_action_entry a, StepOut& o) {
    uint32_t layers = (uint32_t)a.layers[0] | ((uint32_t)a.layers[1] << 8) | ((uint32_t)a.layers[2] << 16) |
                      ((uint32_t)a.layers[3] << 24);
    if (layers == 0) {                       // the common case: no pass-through novelty around this action
        terminal_op(e, cfg, a, o);
        post_step(e, cfg, o);
        return;
    }
    int fr, fc;
    front_of(e, fr, fc);
    int front = cell(e, fr, fc);             // nothing before the terminal opcode changes the grid
    int n = 0, stop = -1;                    // stop = index of the FenceRestriction layer that refused, -1 = none
    for (; n < NGW_MAX_LAYERS; n++) {
        int layer = (layers >> (8 * n)) & 0xFF;
        if (layer == NGW_LAYER_END) break;
        if (layer == NGW_LAYER_CRATE) {                               // novelty_wrappers.py:1085-1088
            if (front == cfg.id_crate)
                for (int it = 0; it < cfg.n_items; it++) inv_add(e, it, (int)cfg.crate_add[it]);
        } else if (layer == NGW_LAYER_FENCE_MEDIUM || layer == NGW_LAYER_FENCE_HARD) {   // novelty_wrappers.py:926-958
            bool pass;
            int fence = cfg.id_fence;
            if (in_mask(cfg.unbreakable_mask, front)) pass = false;
            else if (front == fence) pass = true;
            else if (layer == NGW_LAYER_FENCE_MEDIUM) {
                bool ns = e.facing == NGW_NORTH || e.facing == NGW_SOUTH;
                int a0 = ns ? cell(e, e.r, e.c - 1) : cell(e, e.r - 1, e.c);
                int a1 = ns ? cell(e, e.r, e.c + 1) : cell(e, e.r + 1, e.c);
                pass = !(a0 == fence || a1 == fence);
            } else {
                bool any = false;
                for (int rr = fr - 1; rr <= fr + 1; rr++)
                    for (int cc = fc - 1; cc <= fc + 1; cc++)
                        if (rr >= 0 && rr < e.ms && cc >= 0 && cc < e.ms) any |= cell(e, rr, cc) == fence;
                pass = !any;
            }
            if (!pass) { stop = n; break; }
        }
    }
    int first_post;                           // innermost layer whose post block runs
    if (stop < 0) {
        terminal_op(e, cfg, a, o);
        post_step(e, cfg, o);
        first_post = n - 1;
    } else {
        o.reward = -1; o.result = 0; o.cost = 3600.0f; o.done = 0; o.msg = 0; o.goal = 0;
        first_post = stop;
    }
    for (int i = first_post; i >= 0; i--) {
        int layer = (layers >> (8 * i)) & 0xFF;
        if (layer == NGW_LAYER_FIREWALL) {                            // novelty_wrappers.py:1171-1189
            if (next_to(e, e.r, e.c, cfg.id_fire_wall)) { o.reward = cfg.reward_firewall; o.done = 1; o.msg = NGW_MSG_FIRE_WALL; }
        } else if (layer == NGW_LAYER_FENCE_MEDIUM || layer == NGW_LAYER_FENCE_HARD) {
            // outer post block re-runs and overwrites info (Q5, novelty_wrappers.py:960-973); reward is the inner one
            int reward = o.reward;
            post_step(e, cfg, o);             // sets done / reward_done from the goal test, done = 0 otherwise
            if (!o.done) o.reward = reward;
            o.result = (i == stop) ? 0 : 1;
            o.cost = 3600.0f;
            // the overwritten info carries this wrapper's own message: '' unless it refused (novelty_wrappers.py:955,958)
            o.msg = (i != stop) ? 0 : (in_mask(cfg.unbreakable_mask, front) ? msg_of(NGW_MSG_CANNOT_BREAK, front)
                                                                             : NGW_MSG_FENCE_RESTRICTION);
        }
    }
}

// ------------------------------------------------------------------ LidarInFront (observation_wrappers.py:32-80)
// Device-side companion of an ngw_config, built by ngw_create from the host beam LUT.  Three paths, chosen per config:
//   lines   (8 beams whose LUT is the canonical compass geometry — the reference default): the beams lie on the four
//           lines through the agent (row, column, two diagonals).  Every cell of a line is read once into an occupancy
//           bit mask (fixed trip count = map size, no data-dependent loop), the nearest set bit on either side of the
//           agent is the cell a beam lands on (ffs / clz), and the reported range is the number of cells for axis beams
//           or firstk[cells] for diagonal beams (the first sample k with round(0.71 k) == cells, from the host LUT).
//   fast    (8 beams, factorised unit step x displacement tables, any rotation pattern): pointer-walking beams.
//   generic (any other beam count): int16 linear-offset LUT [4][B][K] in global memory.
#define NGW_MAX_RANGE 96
struct LidarDev {
    int32_t fast;                       // 1 => unit/disp tables are valid
    int32_t lines;                      // 1 => canonical geometry: firstk/rot are valid (line-gather path)
    int16_t unit[4][8];                 // linear offset d_row * ms + d_col of one step of beam b when facing f
    uint8_t disp[2][NGW_MAX_RANGE];     // cells travelled at sample k (0-based) by even / odd beams
    uint8_t firstk[NGW_MAX_MAP_SIZE];   // firstk[d-1]: 1-based sample at which a diagonal beam first reaches its d-th cell, 0 = never
    alignas(4) uint8_t rot[4];          // beam b of an agent facing f looks along compass direction (b + rot[f]) & 7
    int32_t tail_first;                 // >= 0: the observation's inventory tail is the id range tail_first .. + n_inv_obs - 1, -1: table
    const int16_t* lut;                 // generic path: device int16 [4][B][K]
};

struct DevConfig {
    ngw_config c;
    LidarDev lidar;
};

// Byte offset of the int32 inventory tail in a row of layout `fmt` (NGW_OBS_*) for a config of L lidar items, B beams.
__host__ __device__ __forceinline__ int obs_tail_offset(int fmt, int L, int B) {
    return fmt == NGW_OBS_I32 ? 4 * L * B : fmt == NGW_OBS_U8 ? ((L * B + 3) & ~3) : ((2 * B + 3) & ~3);
}

// One env's observation row: lidar part as int32 (the reference's vector), as uint8 (NGW_OBS_U8: ranges are
// <= max_range <= 90, so the narrowing is exact) or as one (item, range) byte pair per beam (NGW_OBS_HITS), followed by
// the int32 inventory tail.  Sinks get a beam's hit as (beam, lidar slot): the hits row stores them apart, the vector
// layouts at beam * L + slot.  Each beam owns its own entry, so warps / lanes sharing a row never touch the same bytes.
struct ObsRow {
    unsigned char* p;
    int fmt;                            // NGW_OBS_I32 / NGW_OBS_U8 / NGW_OBS_HITS
    __device__ __forceinline__ void put(int beam, int slot, int L, int v) const {
        if (fmt == NGW_OBS_I32) reinterpret_cast<int32_t*>(p)[beam * L + slot] = v;
        else if (fmt == NGW_OBS_U8) p[beam * L + slot] = (unsigned char)v;
        else reinterpret_cast<uint16_t*>(p)[beam] = (uint16_t)((slot + 1) | (v << 8));
    }
    __device__ __forceinline__ void put_beam(int, bool hit, int beam, int slot, int L, int v) const {
        if (hit) put(beam, slot, L, v);
    }
    __device__ __forceinline__ int32_t* tail(int L, int B) const {
        return reinterpret_cast<int32_t*>(p + obs_tail_offset(fmt, L, B));
    }
    __device__ __forceinline__ void put_tail(int L, int B, int i, int v) const { tail(L, B)[i] = v; }
};

// Observation "sink" of the closed-loop rollout: instead of materialising the (sparse) observation row and scanning it,
// the integer linear policy  score[a] = bias[a] + sum_j obs[j] * W[j][a]  is accumulated entry by entry as the lidar
// produces them (<= 8 ranges + the inventory tail).  W: [obs_dim][A] int32, staged in shared memory by the kernel.
struct PolicySink {
    const int32_t* w;
    int A;
    int acc[16];
    __device__ __forceinline__ void init(const int32_t* weights, const int32_t* bias, int n_actions) {
        w = weights; A = n_actions;
#pragma unroll
        for (int a = 0; a < 16; a++) acc[a] = a < A ? bias[a] : 0;
    }
    __device__ __forceinline__ void add(int idx, int v) {               // obs[idx] = v
        const int32_t* row = w + idx * A;
#pragma unroll
        for (int a = 0; a < 16; a++) if (a < A) acc[a] += v * row[a];
    }
    __device__ __forceinline__ void put(int beam, int slot, int L, int v) { add(beam * L + slot, v); }
    __device__ __forceinline__ void put_beam(int, bool hit, int beam, int slot, int L, int v) { if (hit) put(beam, slot, L, v); }
    __device__ __forceinline__ void put_tail(int L, int B, int i, int v) { if (v != 0) add(L * B + i, v); }
    __device__ __forceinline__ int argmax(int n_valid) const {       // first maximum over the env's valid action ids
        int best = 0, best_v = acc[0];
#pragma unroll
        for (int a = 1; a < 16; a++) if (a < n_valid && acc[a] > best_v) { best_v = acc[a]; best = a; }
        return best;
    }
};

// Observation sink of the warp-per-tile step kernel (step1w_kernel): the <= 8 lidar hits and the inventory tail stay in
// REGISTERS (every call site has a compile-time beam / tail position) while the observation tile's shared memory is
// still occupied by the grid and inventory rows it aliases; flush() writes them into the zeroed row afterwards.
#define NGW_REGSINK_TAIL 16
template <int NT>
struct RegSink {
    uint32_t hit[8];                    // per compass direction: (beam << 16) | (lidar slot << 8) | range, 0 = nothing seen
    int32_t tail[NT];
    int sh;                             // log2 of the bytes per lidar entry (2: int32 rows, 0: NGW_OBS_U8, 1: NGW_OBS_HITS)
    __device__ __forceinline__ void init(int fmt) {
        sh = fmt == NGW_OBS_I32 ? 2 : fmt == NGW_OBS_U8 ? 0 : 1;
#pragma unroll
        for (int a = 0; a < 8; a++) hit[a] = 0u;
#pragma unroll
        for (int i = 0; i < NT; i++) tail[i] = 0;
    }
    __device__ __forceinline__ void put_beam(int a, bool on, int beam, int slot, int L, int v) {   // every position is written exactly once
        const uint32_t packed = on ? ((uint32_t)beam << 16) | ((uint32_t)slot << 8) | (uint32_t)v : 0u;   // (range >= 1)
#pragma unroll
        for (int j = 0; j < 8; j++) if (j == a) hit[j] = packed;
    }
    __device__ __forceinline__ void put_tail(int, int, int i, int v) {
#pragma unroll
        for (int j = 0; j < NT; j++) if (j == i) tail[j] = v;
    }
    __device__ __forceinline__ void put(int, int, int, int) {}       // (generic LUT walk: never taken with this sink)
    // row: the lane's (zeroed) observation row, dump: a scratch word, both as shared-memory addresses.  Branch-free: a
    // beam that saw nothing and a tail slot beyond n_tail store to the dump word instead.
    // L: lidar items of the lane's config.
    __device__ __forceinline__ void flush(uint32_t row, uint32_t dump, int L, int tail_off, int n_tail) const {
        if (sh == 1) {                                                // (item, range) halfword at byte 2 * beam
#pragma unroll
            for (int a = 0; a < 8; a++)
                asm volatile("st.shared.u16 [%0], %1;" ::"r"(hit[a] ? row + ((hit[a] >> 16) << 1) : dump),
                             "r"(((hit[a] & 0xFFu) << 8) + ((hit[a] >> 8) & 0xFFu) + 1u) : "memory");
        } else {
#pragma unroll
            for (int a = 0; a < 8; a++) {
                const uint32_t off = ((hit[a] >> 16) * (uint32_t)L + ((hit[a] >> 8) & 0xFFu)) << sh;
                if (sh == 2) asm volatile("st.shared.b32 [%0], %1;" ::"r"(hit[a] ? row + off : dump), "r"(hit[a] & 0xFFu) : "memory");
                else asm volatile("st.shared.u8 [%0], %1;" ::"r"(hit[a] ? row + off : dump), "r"(hit[a]) : "memory");
            }
        }
        const uint32_t t = row + (uint32_t)tail_off;
#pragma unroll
        for (int i = 0; i < NT; i++)
            asm volatile("st.shared.b32 [%0], %1;" ::"r"(i < n_tail ? t + 4u * i : dump), "r"(tail[i]) : "memory");
    }
};

// Small per-config lookup tables the lidar reads with per-lane indices (shared memory in the step kernel, global
// memory in the cold kernels): item id -> lidar slot, diagonal cells -> first sample.
struct LidarLuts {
    const int8_t* slot;                 // [NGW_MAX_ITEMS]
    const uint8_t* firstk;              // [NGW_MAX_MAP_SIZE]
};

template <typename MaskT> __device__ __forceinline__ int mask_ffs(MaskT x);
template <> __device__ __forceinline__ int mask_ffs<uint32_t>(uint32_t x) { return __ffs((int)x); }
template <> __device__ __forceinline__ int mask_ffs<uint64_t>(uint64_t x) { return __ffsll((long long)x); }
template <typename MaskT> __device__ __forceinline__ int mask_msb(MaskT x);      // index of the highest set bit, x != 0
template <> __device__ __forceinline__ int mask_msb<uint32_t>(uint32_t x) { return 31 - __clz((int)x); }
template <> __device__ __forceinline__ int mask_msb<uint64_t>(uint64_t x) { return 63 - __clzll((long long)x); }

// occupancy of the four lines through (r, c); bit i = cell of the line in grid row i (row line: grid column i).
// MS > 0 / SEL >= 0 fix the map size / the set of lines at compile time (fully unrolled, immediate offsets, no
// predication); kSafe clamps the diagonal addresses into the row (cold kernels on global memory) — the step kernel's
// shared-memory rows have >= ms bytes of readable padding on both sides, and out-of-grid bits are masked off either way.
template <typename MaskT, int MS, int SEL, bool kSafe>
__device__ __forceinline__ void gather_lines(const int8_t* m, int ms_rt, int r, int c, int sel_rt, MaskT& row, MaskT& col,
                                             MaskT& dg, MaskT& an) {
    const int ms = MS > 0 ? MS : ms_rt;
    const int sel = SEL >= 0 ? SEL : sel_rt;
    const uint8_t* base = reinterpret_cast<const uint8_t*>(m);
    const uint8_t* prow = base + r * ms;
    const uint8_t* pcol = base + c;
    const uint8_t* pdg = base + (c - r);                              // row i: column c - r + i
    const uint8_t* pan = base + (c + r);                              // row i: column c + r - i
    row = 0; col = 0; dg = 0; an = 0;
    if (SEL >= 0) {                                                   // one fused, fully unrolled pass over the chosen lines
#pragma unroll
        for (int i = 0; i < ms; i++) {
            const MaskT bit = (MaskT)1 << i;
            if (sel & 1) { if (prow[i] != 0) row |= bit; }
            if (sel & 2) { if (pcol[i * ms] != 0) col |= bit; }
            if (sel & 4) { if (pdg[i * (ms + 1)] != 0) dg |= bit; }
            if (sel & 8) { if (pan[i * (ms - 1)] != 0) an |= bit; }
        }
    } else {                                                          // any size / any subset: one loop per line, `sel` is warp-uniform
        if (sel & 1) {
#pragma unroll 8
            for (int i = 0; i < ms; i++) if (prow[i] != 0) row |= (MaskT)1 << i;
        }
        if (sel & 2) {
#pragma unroll 8
            for (int i = 0; i < ms; i++) if (pcol[i * ms] != 0) col |= (MaskT)1 << i;
        }
        if (sel & 4) {
#pragma unroll 8
            for (int i = 0; i < ms; i++) {
                int cd = c - r + i;
                if (kSafe) cd = cd < 0 ? 0 : (cd > ms - 1 ? ms - 1 : cd);
                if (base[i * ms + cd] != 0) dg |= (MaskT)1 << i;
            }
        }
        if (sel & 8) {
#pragma unroll 8
            for (int i = 0; i < ms; i++) {
                int ca = c + r - i;
                if (kSafe) ca = ca < 0 ? 0 : (ca > ms - 1 ? ms - 1 : ca);
                if (base[i * ms + ca] != 0) an |= (MaskT)1 << i;
            }
        }
    }
    // rows whose diagonal cell lies outside the grid: r - c <= i <= r - c + ms - 1, resp. c + r - ms + 1 <= i <= c + r
    const MaskT full = (MaskT)(~(MaskT)0) >> (8 * (int)sizeof(MaskT) - ms);
    const int dlo = r - c, alo = c + r - (ms - 1);
    dg &= dlo >= 0 ? (full << dlo) : (full >> (-dlo));
    an &= alo >= 0 ? (full << alo) : (full >> (-alo));
}

// the two beams of one line: `p` = the agent's bit index on the line, `stride` = linear offset of one cell towards
// higher bit indices, a_pos / a_neg = compass directions of the two beams
template <typename MaskT, typename Sink>
__device__ __forceinline__ void line_beams(MaskT occ, int p, int stride, const int8_t* here, bool diagonal, int a_pos,
                                           int a_neg, int K, int L, int rot, const LidarLuts& luts, Sink& obs) {
    const MaskT hi = (occ >> p) >> 1;                                 // bit 0 = the cell next to the agent
    const MaskT lo = occ & (((MaskT)1 << p) - 1);
    const int n_pos = mask_ffs<MaskT>(hi);                            // cells to the first non-air cell, 0 = none
    const int n_neg = lo != 0 ? p - mask_msb<MaskT>(lo) : 0;
    // no early-outs: a beam that sees nothing (n == 0) reads the agent's own cell — air, whose slot is -1
#pragma unroll
    for (int side = 0; side < 2; side++) {
        const int n = side ? n_neg : n_pos;
        const int a = side ? a_neg : a_pos;
        const int k = diagonal ? (int)luts.firstk[n - 1] : (n <= K ? n : 0);   // obsw:52-58: sample index of that cell, 0 = beyond max_beam_range
        const int id = here[side ? -n * stride : n * stride];
        const int slot = luts.slot[id];                               // -1: occludes but is not a lidar item (Q2)
        obs.put_beam(a, slot >= 0 && n != 0 && k != 0, (a - rot) & 7, slot, L, k);
    }
}

template <typename MaskT, int MS, int SEL, bool kSafe, typename Sink>
__device__ __forceinline__ void lidar_lines_t(const EnvRow& e, const ngw_config& cfg, const LidarDev& t,
                                              const LidarLuts& luts, Sink& obs, int sel_rt) {
    MaskT row, col, dg, an;
    gather_lines<MaskT, MS, SEL, kSafe>(e.m, e.ms, e.r, e.c, sel_rt, row, col, dg, an);
    const int ms = MS > 0 ? MS : e.ms;
    const int sel = SEL >= 0 ? SEL : sel_rt;
    const int K = cfg.max_range, L = cfg.n_lidar_items;
    const int rot = (int)((*reinterpret_cast<const uint32_t*>(t.rot) >> (8 * e.facing)) & 7u);   // one uniform table read
    const int8_t* here = e.m + e.r * ms + e.c;
    // compass directions (d_row, d_col): 0 (+1,0)  1 (+1,+1)  2 (0,+1)  3 (-1,+1)  4 (-1,0)  5 (-1,-1)  6 (0,-1)  7 (+1,-1)
    if (sel & 1) line_beams<MaskT, Sink>(row, e.c, 1, here, false, 2, 6, K, L, rot, luts, obs);
    if (sel & 2) line_beams<MaskT, Sink>(col, e.r, ms, here, false, 0, 4, K, L, rot, luts, obs);
    if (sel & 4) line_beams<MaskT, Sink>(dg, e.r, ms + 1, here, true, 1, 5, K, L, rot, luts, obs);
    if (sel & 8) line_beams<MaskT, Sink>(an, e.r, ms - 1, here, true, 7, 3, K, L, rot, luts, obs);
}

// `sel` is warp-uniform.  The hot shapes (the reference's 10x10 grid; all four lines, or the axis / diagonal halves of
// a two-warp tile) get fully unrolled, unpredicated code; other sizes share two generic loops.  (Grids above 32x32 keep
// the pointer-walking beams, see lidar_observe: on C5's dense 40x40 grids beams land after a few cells, and reading whole
// 40-cell lines — or 16-cell windows outwards, also tried — measured 2-8 % slower than walking.)
template <bool kSafe, typename Sink>
__device__ __forceinline__ void lidar_lines(const EnvRow& e, const ngw_config& cfg, const LidarDev& t,
                                            const LidarLuts& luts, Sink& obs, int sel) {
    if (!kSafe && e.ms == 10 && sel == 0xF) lidar_lines_t<uint32_t, 10, 0xF, false, Sink>(e, cfg, t, luts, obs, sel);
    else if (!kSafe && e.ms == 10 && sel == 0x3) lidar_lines_t<uint32_t, 10, 0x3, false, Sink>(e, cfg, t, luts, obs, sel);
    else if (!kSafe && e.ms == 10 && sel == 0xC) lidar_lines_t<uint32_t, 10, 0xC, false, Sink>(e, cfg, t, luts, obs, sel);
    else if (e.ms <= 32) lidar_lines_t<uint32_t, 0, -1, kSafe, Sink>(e, cfg, t, luts, obs, sel);
    else lidar_lines_t<uint64_t, 0, -1, kSafe, Sink>(e, cfg, t, luts, obs, sel);
}

// which of the four lines warp g of G handles (bit 0 row, 1 column, 2 diagonal, 3 anti-diagonal)
__device__ __forceinline__ int lidar_line_share(int g, int G) {
    if (G == 1) return 0xF;
    if (G == 2) return g == 0 ? 0x3 : 0xC;
    return g < 4 ? (1 << g) : 0;
}

// obs row must be zero-filled for the lidar part by the caller; `zero` points at a byte that always reads 0 and lives in
// the same address space as the grid row.  A tile can be shared by G warps: warp `g` of `G` casts beams
// [g*NB, (g+1)*NB) with NB = 8/G (fast path) or beams g, g+G, ... (generic path).
template <int NB, typename Sink>
__device__ __forceinline__ void lidar_fast(const EnvRow& e, const ngw_config& cfg, const LidarDev& lidar, Sink& obs,
                                           const int8_t* zero, int b0) {
    // Each beam keeps a running cell pointer; axis beams advance one unit step per sample, diagonal beams advance
    // when round(0.71 k) grows (disp[1][k] - disp[1][k-1] is 0 or 1).  A beam that lands parks on `zero`, a cell
    // that always reads air, so no per-beam "still flying" test is needed in the loop.
    const int K = cfg.max_range, L = cfg.n_lidar_items;
    int u[NB];
    const int8_t* at[NB];
    uint32_t hit[NB];                                                 // (sample index << 8) | item id, 0 = still flying
    const int8_t* base = e.m + e.r * e.ms + e.c;
#pragma unroll
    for (int j = 0; j < NB; j++) { u[j] = lidar.unit[e.facing][b0 + j]; at[j] = base; hit[j] = 0; }
    int prev0 = 0, prev1 = 0, flying = 1;                             // a unit step is never 0, so OR(u) != 0 <=> a beam still flies
    for (int k = 0; k < K && flying != 0; k++) {
        const int d0 = lidar.disp[0][k], d1 = lidar.disp[1][k];
        const int s0 = d0 - prev0, s1 = d1 - prev1;                   // warp-uniform step counts (0 or 1 for 8 beams)
        prev0 = d0; prev1 = d1;
        int id[NB];
#pragma unroll
        for (int j = 0; j < NB; j++) {                                // NB independent shared-memory reads in flight
            at[j] += u[j] * (((b0 + j) & 1) ? s1 : s0);
            id[j] = *at[j];
        }
#pragma unroll
        for (int j = 0; j < NB; j++) {
            bool lands = id[j] != 0;                                  // first non-air cell ends the beam (obsw:58-66)
            hit[j] = lands ? (uint32_t)(((k + 1) << 8) | (id[j] & 0xFF)) : hit[j];
            u[j] = lands ? 0 : u[j];
            at[j] = lands ? zero : at[j];
        }
        flying = 0;
#pragma unroll
        for (int j = 0; j < NB; j++) flying |= u[j];
    }
#pragma unroll
    for (int j = 0; j < NB; j++) {                                    // (sinks with positions: j-th beam of this warp's share)
        const int slot = hit[j] ? (int)cfg.lidar_slot[hit[j] & 0xFF] : -1;   // -1: occludes but is not a lidar item (Q2)
        obs.put_beam(j, slot >= 0, b0 + j, slot, L, (int)(hit[j] >> 8));
    }
}

// inventory tail of the observation (observation_wrappers.py:77-78): quantities in sorted-name order minus unbreakables (Q7)
// tail_first: LidarDev::tail_first of the env's config.  Item ids follow the sorted names (pogostick_v1_env.py:200-212),
// so without late-injected items the tail is an id range and the copy needs no table; NT bounds the unrolled copy.
template <typename Sink, int NT = 16>
__device__ __forceinline__ void obs_tail(const EnvRow& e, const ngw_config& cfg, Sink& obs, int tail_first) {
    const int n_tail = cfg.n_inv_obs, L = cfg.n_lidar_items, B = cfg.n_beams;
    if (tail_first >= 0 && n_tail <= NT) {
        const int32_t* src = e.inv + tail_first;
#pragma unroll
        for (int i = 0; i < NT; i++) if (i < n_tail) obs.put_tail(L, B, i, src[i]);
        return;
    }
    for (int i = 0; i < n_tail; i++) obs.put_tail(L, B, i, e.inv[cfg.inv_obs_item[i]]);
}

// `tables`: the beam tables to walk with — the env's own config, or (mixed batches whose configs all share one lidar
// geometry) config 0's, so that the table reads stay warp-uniform even when the lanes of a warp differ in config.
// `luts` (line path only): where the per-lane indexed slot / firstk tables live; luts.slot == nullptr selects the
// pointer-walking path even when the geometry is canonical.
template <bool kSafe, typename Sink = ObsRow>
__device__ __forceinline__ void lidar_observe(const EnvRow& e, const DevConfig& dc, const LidarDev& tables,
                                              const LidarLuts& luts, Sink& obs, const int8_t* zero, int g, int G,
                                              bool with_tail) {
    const ngw_config& cfg = dc.c;
    const int B = cfg.n_beams, K = cfg.max_range, L = cfg.n_lidar_items;
    // (`lines` implies `fast`, so `!fast` never holds here; written out, it keeps observe_masked_kernel at 62 registers
    // instead of 68 and rollout_kernel's spills where they were)
    if (dc.lidar.lines && luts.slot != nullptr && (e.ms <= 32 || !dc.lidar.fast)) {
        const int sel = lidar_line_share(g, G);
        if (sel) lidar_lines<kSafe, Sink>(e, cfg, tables, luts, obs, sel);
    } else if (dc.lidar.fast) {
        if (G == 1) lidar_fast<8, Sink>(e, cfg, tables, obs, zero, 0);
        else if (G == 2) lidar_fast<4, Sink>(e, cfg, tables, obs, zero, g * 4);
        else if (G == 4) lidar_fast<2, Sink>(e, cfg, tables, obs, zero, g * 2);
        else lidar_fast<1, Sink>(e, cfg, tables, obs, zero, g);         // G == 8: the reset kernel's observation pass
    } else {
        const int cells = e.ms * e.ms;
        const int pos = e.r * e.ms + e.c;
        for (int b = g; b < B; b += G) {
            const int16_t* row = dc.lidar.lut + (e.facing * B + b) * K;
            for (int k = 0; k < K; k++) {
                int idx = pos + row[k];
                if ((unsigned)idx >= (unsigned)cells) break;
                int id = e.m[idx];
                if (id != 0) {
                    int slot = cfg.lidar_slot[id];
                    if (slot >= 0) obs.put(b, slot, L, k + 1);
                    break;
                }
            }
        }
    }
    if (with_tail) obs_tail<Sink>(e, cfg, obs, dc.lidar.tail_first);
}

// ------------------------------------------------------------------ reset (pogostick_v1_env.py:86-181 + novelty resets)
// WARP-COOPERATIVE: the 32 lanes of one warp regenerate ONE environment (rows in shared or global memory).
//
// Same DISTRIBUTION as the reference, not the same stream (reset_env_numpy_warp below draws the reference's own stream):
//  * placement: the reference draws uniformly from a list it shrinks by popping every drawn cell; a popped cell is the
//    agent cell, a placed item or a cell that can never become placeable again, so "first placeable cell in a uniformly
//    random order" == uniform over the currently placeable cells == draw-with-replacement-until-placeable (no list).
//    These few draws are computed redundantly by all lanes (identical Philox counters), lane 0 writes.
//  * post-ops ("shuffle the candidate cells, take the first m", m = ceil(n * (pct / 100)) in IEEE doubles as NumPy does):
//    a uniformly random m-subset.  Every candidate cell gets an independent 32-bit Philox key (counter = cell index) and
//    the m smallest keys win — found with a warp radix-select (256-bin histogram in shared memory) and, inside the
//    boundary bin, an exact rank by (key, cell index), so equal keys go by cell index.  Only when more than 32 candidates
//    share the boundary key exactly (probability ~ n^2 / 2^33) do they win in arrival order instead, which is
//    (i >> 7, i & 3, i >> 2) for cell i: 128-cell rounds, then the word of the key's Philox block, then the lane.
__device__ __forceinline__ bool placeable(const int8_t* m, int ms, int r, int c) {
    const int8_t* p = m + r * ms + c;
    return p[0] == 0 && p[-ms] == 0 && p[ms] == 0 && p[-1] == 0 && p[1] == 0;
}

// keys of the four cells 4q .. 4q+3: one Philox block (block 0 of the stream draws the percentage)
__device__ __forceinline__ void philox_keys4(uint64_t seed, uint64_t gid, uint32_t episode, uint32_t stream, uint32_t q,
                                             uint32_t key[4]) {
    Philox rng;
    rng.init(seed, gid, episode, stream);
    rng.blk = 1 + q;
    rng.refill();
    key[0] = rng.buf[0]; key[1] = rng.buf[1]; key[2] = rng.buf[2]; key[3] = rng.buf[3];
}

__device__ __forceinline__ bool reset_candidate(int kind, int id, int wall, int a) {
    return kind == NGW_RESET_FENCE ? (id != 0 && id != wall)           // novelty_wrappers.py:872
         : kind == NGW_RESET_ADDITEM ? (id == 0)                       // novelty_wrappers.py:1017
         : (id == a);                                                  // novelty_wrappers.py:1130
}

// The 32 lanes of one warp regenerate one environment (ngw_reset, the queued auto-resets, the in-place regeneration of
// the rollout kernels).  All lanes call with the same arguments.  `hist`: NGW_RESET_SCRATCH_WORDS uint32 of shared
// memory owned by the warp.
#define NGW_RESET_SCRATCH_WORDS (256 + 32)
static __device__ __noinline__ uint32_t reset_env_warp(const ngw_config* cfg, int8_t* m, int32_t* inv, int ms, int inv_stride,
                                                       uint64_t seed, uint64_t gid, uint32_t episode, bool do_base,
                                                       int op_begin, int op_end, uint32_t* hist, int& pr, int& pc, int& pf,
                                                       int& psel, uint32_t key_mask = 0xFFFFFFFFu) {
    const uint32_t FULL = 0xFFFFFFFFu;
    const int lane = threadIdx.x & 31;
    uint32_t* xw = hist + 256;                                        // [1] boundary-list length, [2..4] scan result
    const int cells = ms * ms;
    const int wall = cfg->id_wall;
    uint32_t err = 0;
    if (do_base) {
        for (int i = lane; i < inv_stride; i += 32) inv[i] = 0;         // pogostick_v1_env.py:119-120
        psel = 0;
        for (int r = lane / ms, c = lane - (lane / ms) * ms, i = lane; i < cells; i += 32) {   // pogostick_v1_env.py:129-130
            m[i] = (r == 0 || c == 0 || r == ms - 1 || c == ms - 1) ? (int8_t)wall : (int8_t)0;
            c += 32;
            while (c >= ms) { c -= ms; r++; }
        }
        __syncwarp();
        Philox rng;
        rng.init(seed, gid, episode, 0);
        const int side = ms - 4;                                      // rows/cols 2 .. ms-3 (pogostick_v1_env.py:136-138)
        const uint32_t n_av = (uint32_t)(side * side);
        uint32_t a = rng.below(n_av);
        pr = 2 + (int)(a / side); pc = 2 + (int)(a % side);           // pogostick_v1_env.py:141-142
        pf = (int)rng.below(4);                                       // pogostick_v1_env.py:145
        const int agent = pr * ms + pc;
        for (int i = 0; i < cfg->n_place; i++) {                      // pogostick_v1_env.py:147-148,159-181
            const int item = cfg->place_item[i], qty = cfg->place_qty[i];
            for (int count = 0; count < qty; count++) {
                int where = -1;
                for (uint32_t attempt = 0; attempt < 8 * n_av && where < 0; attempt++) {
                    uint32_t d = rng.below(n_av);
                    int r = 2 + (int)(d / side), c = 2 + (int)(d % side);
                    if (r * ms + c != agent && placeable(m, ms, r, c)) where = r * ms + c;
                }
                if (where < 0) {                                      // rare: enumerate the placeable cells exactly
                    uint32_t good = 0;
                    for (int r = 2; r <= ms - 3; r++)
                        for (int c = 2; c <= ms - 3; c++) good += (r * ms + c != agent && placeable(m, ms, r, c));
                    if (good == 0) { err |= NGW_ERR_PLACEMENT; i = cfg->n_place; break; }   // pogostick_v1_env.py:167
                    uint32_t pick = rng.below(good);
                    for (int r = 2; r <= ms - 3 && where < 0; r++)
                        for (int c = 2; c <= ms - 3 && where < 0; c++)
                            if (r * ms + c != agent && placeable(m, ms, r, c)) {
                                if (pick == 0) where = r * ms + c;
                                pick--;
                            }
                }
                __syncwarp();                                         // every lane has read the grid it decided on
                if (lane == 0) m[where] = (int8_t)item;
                __syncwarp();
            }
        }
    }
    const int agent = pr * ms + pc;
    if (op_end > cfg->n_reset_ops) op_end = cfg->n_reset_ops;
    for (int k = op_begin; k < op_end; k++) {
        const ngw_reset_op op = cfg->reset_ops[k];
        if (op.kind == NGW_RESET_INVSET) {                            // novelty_wrappers.py:33,460,668-671
            if (lane == 0) inv[op.a] = op.lo;
            __syncwarp();
            continue;
        }
        const uint32_t stream = 1 + k;
        if (op.kind == NGW_RESET_TREETAP) {                           // pogostick_v0_env.py:155-178
            // uniform over (tree_log, direction) pairs until the target cell is free == the reference's retry loop;
            // done by the whole warp (a rare op on 10x10 grids), the draws redundantly by its lanes
            int target = -1, n_logs = 0;
            for (int i = lane; i < cells; i += 32) n_logs += (m[i] == (int8_t)op.b);
            n_logs = __reduce_add_sync(FULL, n_logs);
            if (n_logs > 1) {
                Philox rt;
                rt.init(seed, gid, episode, stream);
                for (int attempt = 0; attempt < 4096 && target < 0; attempt++) {
                    int direction = (int)rt.below(4);
                    int which = (int)rt.below((uint32_t)n_logs);
                    int log = -1;
                    for (int base = 0; base < cells && log < 0; base += 32) {     // which-th tree_log in row-major order
                        int i = base + lane;
                        uint32_t bal = __ballot_sync(FULL, i < cells && m[i] == (int8_t)op.b);
                        int c = __popc(bal);
                        if (which < c) {
                            int bit = __fns(bal, 0, which + 1);
                            log = base + bit;
                        } else which -= c;
                    }
                    int r = log / ms, c = log - r * ms;
                    int tr = r + (direction == NGW_SOUTH) - (direction == NGW_NORTH);
                    int tc = c + (direction == NGW_EAST) - (direction == NGW_WEST);
                    if (tr >= 0 && tr < ms && tc >= 0 && tc < ms && m[tr * ms + tc] == 0 && tr * ms + tc != agent)
                        target = tr * ms + tc;
                }
            }
            if (lane == 0) { xw[2] = (uint32_t)n_logs; xw[3] = (uint32_t)target; }
            __syncwarp();
            n_logs = (int)xw[2]; target = (int)xw[3];
            __syncwarp();
            if (n_logs <= 1 || target < 0) { err |= NGW_ERR_PLACEMENT; continue; }
            if (lane == 0) m[target] = (int8_t)op.a;
            __syncwarp();
            continue;
        }
        // ---- n candidates, percentage, m
        int n = 0;
        for (int i = lane; i < cells; i += 32) n += reset_candidate(op.kind, m[i], wall, op.a);
        n = __reduce_add_sync(FULL, n);
        Philox rng;
        rng.init(seed, gid, episode, stream);
        const int pct = op.lo + (int)rng.below((uint32_t)(op.hi - op.lo));            // randint(low, high), high exclusive
        int take = (int)ceil((double)n * ((double)pct / 100.0));                      // novelty_wrappers.py:881,1025,1139
        if (take > n) take = n;
        if (take <= 0) continue;
        // ---- radix-select the `take` smallest keys: after the loop, keys whose top `bits` bits are < prefix win outright,
        //      keys whose top bits == prefix compete for the `remaining` last places
        uint32_t prefix = 0;
        int bits = 0, remaining = take, bin_count = n;
        const int quads = (cells + 3) >> 2;                           // a thread handles 4 consecutive cells per Philox block
        while (remaining < bin_count && bin_count > 32 && bits < 32) {
            for (int i = lane; i < 256; i += 32) hist[i] = 0;
            __syncwarp();
            for (int q = lane; q < quads; q += 32) {
                bool cand[4], any = false;
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    int i = 4 * q + j;
                    cand[j] = i < cells && reset_candidate(op.kind, m[i < cells ? i : 0], wall, op.a);
                    any |= cand[j];
                }
                if (!any) continue;
                uint32_t key[4];
                philox_keys4(seed, gid, episode, stream, (uint32_t)q, key);
#pragma unroll
                for (int j = 0; j < 4; j++) key[j] &= key_mask;
#pragma unroll
                for (int j = 0; j < 4; j++)
                    if (cand[j] && (bits == 0 || (key[j] >> (32 - bits)) == prefix))
                        atomicAdd(&hist[(key[j] >> (24 - bits)) & 0xFF], 1u);
            }
            __syncwarp();
            uint32_t mine[8], sum = 0;                                // scan the 256 bins, 8 per lane
#pragma unroll
            for (int j = 0; j < 8; j++) { mine[j] = hist[lane * 8 + j]; sum += mine[j]; }
            uint32_t incl = sum;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                uint32_t t = __shfl_up_sync(FULL, incl, o);
                if (lane >= o) incl += t;
            }
            uint32_t excl = incl - sum;
            bool owner = (uint32_t)remaining > excl && (uint32_t)remaining <= incl;   // the bin holding the remaining-th key
            if (owner) {
                uint32_t below = excl;
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    if ((uint32_t)remaining <= below + mine[j]) { xw[2] = (uint32_t)(lane * 8 + j); xw[3] = below; xw[4] = mine[j]; break; }
                    below += mine[j];
                }
            }
            __syncwarp();
            const uint32_t bin = xw[2], below = xw[3], cnt = xw[4];
            __syncwarp();
            prefix = (prefix << 8) | bin;
            bits += 8;
            remaining -= (int)below;
            bin_count = (int)cnt;
        }
        // ---- apply: one pass; winners are written at once, boundary-bin cells (<= 32, unless all of them win) are listed
        const bool all_in_bin_win = remaining >= bin_count;
        const bool exact_keys = bits >= 32 && bin_count > 32;
        const int value = op.kind == NGW_RESET_ADDITEM ? op.a : op.b;
        if (lane == 0) xw[1] = 0;
        __syncwarp();
        for (int qb = 0; qb < quads; qb += 32) {
            const int q = qb + lane;
            uint32_t key[4] = {0, 0, 0, 0};
            int id[4]; bool cand[4], any = false;
#pragma unroll
            for (int j = 0; j < 4; j++) {
                int i = 4 * q + j;
                id[j] = (q < quads && i < cells) ? (int)m[i] : 0;
                cand[j] = q < quads && i < cells && reset_candidate(op.kind, id[j], wall, op.a);
                any |= cand[j];
            }
            if (any) philox_keys4(seed, gid, episode, stream, (uint32_t)q, key);
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const int i = 4 * q + j;
                key[j] &= key_mask;
                uint32_t top = bits == 0 ? 0 : (key[j] >> (32 - bits));
                bool wins = cand[j] && (bits == 0 ? all_in_bin_win : (top < prefix || (top == prefix && all_in_bin_win)));
                bool boundary = cand[j] && !all_in_bin_win && top == prefix;
                uint32_t bal = __ballot_sync(FULL, boundary);
                if (bal != 0) {
                    // a slot per boundary cell: warp-aggregated counter in shared memory (the list is ranked by
                    // (key, cell) afterwards)
                    int base = 0;
                    if (lane == __ffs((int)bal) - 1) base = (int)atomicAdd(&xw[1], (uint32_t)__popc(bal));
                    base = __shfl_sync(FULL, base, __ffs((int)bal) - 1);
                    if (boundary) {
                        int slot = base + __popc(bal & ((1u << lane) - 1u));
                        // all 32 key bits consumed and still more than 32 contenders: their keys are IDENTICAL (probability
                        // ~ n^2 / 2^33 per reset), so the tie goes by arrival order and no list is needed
                        if (exact_keys) wins = slot < remaining;
                        else if (slot < 32) { hist[slot] = key[j]; hist[32 + slot] = (uint32_t)i; }
                    }
                }
                if (wins) {
                    if (op.kind == NGW_RESET_FENCE) m[i] = (int8_t)(id[j] | 0x80);    // mark; fences go in afterwards
                    else if (i != agent) m[i] = (int8_t)value;                        // novelty_wrappers.py:1027,1141
                }
            }
        }
        __syncwarp();
        int n_list = (int)xw[1];
        if (n_list > 0 && !exact_keys) {
            if (n_list > 32) n_list = 32;                             // unreachable: the loop above ends with <= 32 contenders or exact keys
            uint32_t my_key = 0; int my_idx = -1;
            if (lane < n_list) { my_key = hist[lane]; my_idx = (int)hist[32 + lane]; }
            int rank = 0;
            for (int j = 0; j < n_list; j++) {
                uint32_t kj = __shfl_sync(FULL, my_key, j);
                int ij = __shfl_sync(FULL, my_idx, j);
                rank += (kj < my_key) || (kj == my_key && ij < my_idx);
            }
            if (lane < n_list && rank < remaining) {
                if (op.kind == NGW_RESET_FENCE) m[my_idx] = (int8_t)(m[my_idx] | 0x80);
                else if (my_idx != agent) m[my_idx] = (int8_t)value;
            }
        }
        __syncwarp();
        if (op.kind == NGW_RESET_FENCE) {                             // add_fence_around, pogostick_v1_env.py:524-536
            // two phases so that the lanes do not race: read every mark first, then write the fences
            for (int i = lane; i < cells; i += 32) {
                int v = m[i];
                if (!(v & 0x80)) continue;
                int r = i / ms, c = i - r * ms;
                for (int rr = r - 1; rr <= r + 1; rr++)
                    for (int cc = c - 1; cc <= c + 1; cc++)
                        if (rr >= 0 && rr < ms && cc >= 0 && cc < ms && m[rr * ms + cc] == 0 && rr * ms + cc != agent)
                            m[rr * ms + cc] = (int8_t)op.a;
            }
            __syncwarp();
            for (int i = lane; i < cells; i += 32) {
                int v = m[i];
                if (v & 0x80) m[i] = (int8_t)(v & 0x7F);
            }
            __syncwarp();
        }
    }
    return err;
}

// ------------------------------------------------------------------ reset with the reference's own stream (NGW_RNG_NUMPY)
// The same program as ngo_reset_legacy (oracle/ngw_oracle.c), draw for draw, on the env's persistent legacy np.random
// state: MT19937 key[624] + pos in global memory, numpy's get_state() layout.  One warp per env; lane l holds the tempered
// output of word wbase + l, and every draw is broadcast with a shuffle, so all lanes take the same (sequential) decisions.
#define NGW_MT_WORDS 624
// TREETAP attempts before the numpy reset gives up with NGW_ERR_PLACEMENT.  The reference retries forever; when at least
// one target is free an attempt finds one with probability >= 1 / (4 ms^2), so with the cap's 2^20 attempts a 40x40
// grid stops early with probability below e^-163.  Only a grid where no log has a free neighbour reaches it.
#define NGW_NUMPY_TREETAP_CAP (1 << 20)

// MT19937 twist: key[i] for i in [a, b) from key[i + o], key[i], key[i + 1]; every lane reads before any lane writes
__device__ __forceinline__ void mt_twist_span(uint32_t* key, int a, int b, int o, int lane) {
    for (int base = a; base < b; base += 32) {
        const int i = base + lane;
        uint32_t v = 0;
        if (i < b) {
            const uint32_t y = (key[i] & 0x80000000u) | (key[i + 1] & 0x7fffffffu);
            v = key[i + o] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
        }
        __syncwarp();
        if (i < b) key[i] = v;
        __syncwarp();
    }
}
// mt_refill (oracle/ngw_oracle.c) in phases whose reads are complete before they start: [0, 227) reads words >= 397,
// [227, 454) and [454, 623) read words 227 back, which the previous phase wrote; word 623 last
static __device__ __noinline__ void mt_twist(uint32_t* key, int lane) {
    mt_twist_span(key, 0, 227, 397, lane);
    mt_twist_span(key, 227, 454, -227, lane);
    mt_twist_span(key, 454, 623, -227, lane);
    if (lane == 0) {
        const uint32_t y = (key[623] & 0x80000000u) | (key[0] & 0x7fffffffu);
        key[623] = key[396] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
    }
    __syncwarp();
}

struct MtWarp {
    uint32_t* key;   // the env's 624 words (global memory)
    int pos;         // next word, 624 = twist first
    int wbase;       // first word of the lanes' window
    uint32_t win;    // lane l: tempered key[wbase + l]

    __device__ __forceinline__ uint32_t next(int lane) {
        if (pos == NGW_MT_WORDS) { mt_twist(key, lane); pos = 0; wbase = -64; }
        if (pos - wbase >= 32) {
            wbase = pos;
            uint32_t y = pos + lane < NGW_MT_WORDS ? key[pos + lane] : 0u;
            y ^= (y >> 11);
            y ^= (y << 7) & 0x9d2c5680u;
            y ^= (y << 15) & 0xefc60000u;
            y ^= (y >> 18);
            win = y;
        }
        return __shfl_sync(0xFFFFFFFFu, win, pos++ - wbase);
    }
    // uniform in [0, max]: masked rejection on 32-bit outputs (legacy random_interval)
    __device__ __forceinline__ uint32_t interval(uint32_t max, int lane) {
        if (max == 0) return 0;
        uint32_t mask = max;
        mask |= mask >> 1; mask |= mask >> 2; mask |= mask >> 4; mask |= mask >> 8; mask |= mask >> 16;
        uint32_t v;
        do { v = next(lane) & mask; } while (v > max);
        return v;
    }
    // np.random.randint(lo, hi) / np.random.choice(hi) with lo = 0
    __device__ __forceinline__ uint32_t randint(uint32_t lo, uint32_t hi, int lane) { return lo + interval(hi - 1u - lo, lane); }
};

// list.pop(idx) on the warp's shared-memory list of n entries
__device__ __forceinline__ void list_pop(uint16_t* list, int idx, int n, int lane) {
    for (int base = idx; base < n - 1; base += 32) {
        const int i = base + lane;
        const uint16_t v = i < n - 1 ? list[i + 1] : (uint16_t)0;
        __syncwarp();
        if (i < n - 1) list[i] = v;
        __syncwarp();
    }
}

// The 32 lanes of one warp regenerate one env from its np.random state (key[624] and *pos_io, global memory) exactly as
// the reference does under that state.  Arguments as reset_env_warp's; `list`: ms * ms uint16 of shared memory owned by
// the warp (the reference's candidate lists).  A placement that runs out of cells, or a TREETAP with no log to tap (or
// past NGW_NUMPY_TREETAP_CAP attempts), returns NGW_ERR_PLACEMENT and skips the rest of the program, as the reference's
// AssertionError does; the caller skips a second part too.  *pos_io is written back in every case.
static __device__ __noinline__ uint32_t reset_env_numpy_warp(const ngw_config* cfg, int8_t* m, int32_t* inv, int ms,
                                                             int inv_stride, uint32_t* key, int32_t* pos_io, bool do_base,
                                                             int op_begin, int op_end, uint16_t* list, int& pr, int& pc,
                                                             int& pf, int& psel) {
    const uint32_t FULL = 0xFFFFFFFFu;
    const int lane = threadIdx.x & 31;
    const int cells = ms * ms;
    const int wall = cfg->id_wall;
    MtWarp mt;
    mt.key = key; mt.pos = *pos_io; mt.wbase = -64; mt.win = 0;
    uint32_t err = 0;
    if (do_base) {                                                    // pogostick_v1_env.py:118-157
        for (int i = lane; i < inv_stride; i += 32) inv[i] = 0;
        psel = 0;
        for (int r = lane / ms, c = lane - (lane / ms) * ms, i = lane; i < cells; i += 32) {
            m[i] = (r == 0 || c == 0 || r == ms - 1 || c == ms - 1) ? (int8_t)wall : (int8_t)0;
            c += 32;
            while (c >= ms) { c -= ms; r++; }
        }
        const int side = ms - 4;                                      // interior cells 2 .. ms-3, row-major
        int n = side * side;
        for (int i = lane; i < n; i += 32) list[i] = (uint16_t)((2 + i / side) * ms + 2 + i % side);
        __syncwarp();
        const int a = (int)mt.randint(0, (uint32_t)n, lane);          // agent cell (stays in the list)
        pr = 2 + a / side; pc = 2 + a % side;
        pf = (int)mt.randint(0, 4, lane);                             // choice(['NORTH','SOUTH','WEST','EAST'])
        const int agent = pr * ms + pc;
        for (int i = 0; i < cfg->n_place && err == 0; i++) {         // add_item_to_map, pogostick_v1_env.py:159-181
            const int item = cfg->place_item[i], qty = cfg->place_qty[i];
            for (int count = 0; count != qty;) {
                if (n < 1) { err = NGW_ERR_PLACEMENT; break; }
                const int idx = (int)mt.randint(0, (uint32_t)n, lane);
                const int cell = list[idx];
                const int r = cell / ms, c = cell - r * ms;
                const bool put = cell != agent && placeable(m, ms, r, c);
                __syncwarp();
                if (put && lane == 0) m[cell] = (int8_t)item;
                __syncwarp();
                count += put;
                list_pop(list, idx, n, lane);                         // popped whether or not the cell was taken
                n--;
            }
        }
    }
    const int agent = pr * ms + pc;
    if (op_end > cfg->n_reset_ops) op_end = cfg->n_reset_ops;
    for (int k = op_begin; k < op_end && err == 0; k++) {
        const ngw_reset_op op = cfg->reset_ops[k];
        if (op.kind == NGW_RESET_INVSET) {
            if (lane == 0) inv[op.a] = op.lo;
            __syncwarp();
            continue;
        }
        if (op.kind == NGW_RESET_TREETAP) {                           // pogostick_v0_env.py:155-178
            int n_logs = 0, target = -1;
            for (int i = lane; i < cells; i += 32) n_logs += (m[i] == (int8_t)op.b);
            n_logs = __reduce_add_sync(FULL, n_logs);
            if (n_logs <= 1) { err = NGW_ERR_PLACEMENT; break; }      // assert len(result[0]) > 1
            for (int attempt = 0; attempt < NGW_NUMPY_TREETAP_CAP && target < 0; attempt++) {
                const int direction = (int)mt.randint(0, 4, lane);
                int which = (int)mt.randint(0, (uint32_t)n_logs, lane);
                int log = -1;
                for (int base = 0; base < cells && log < 0; base += 32) {   // which-th tree_log in row-major order
                    const int i = base + lane;
                    const uint32_t bal = __ballot_sync(FULL, i < cells && m[i] == (int8_t)op.b);
                    const int cnt = __popc(bal);
                    if (which < cnt) log = base + (int)__fns(bal, 0, which + 1);
                    else which -= cnt;
                }
                const int r = log / ms, c = log - r * ms;
                const int tr = r + (direction == NGW_SOUTH) - (direction == NGW_NORTH);
                const int tc = c + (direction == NGW_EAST) - (direction == NGW_WEST);
                if (tr >= 0 && tr < ms && tc >= 0 && tc < ms && m[tr * ms + tc] == 0 && tr * ms + tc != agent)
                    target = tr * ms + tc;
            }
            if (target < 0) { err = NGW_ERR_PLACEMENT; break; }
            __syncwarp();
            if (lane == 0) m[target] = (int8_t)op.a;
            __syncwarp();
            continue;
        }
        // FENCE / ADDITEM / REPLACE: candidates in row-major order (np.where), shuffled whole, THEN the percentage
        int n = 0;
        for (int base = 0; base < cells; base += 32) {
            const int i = base + lane;
            const bool cand = i < cells && reset_candidate(op.kind, m[i], wall, op.a);
            const uint32_t bal = __ballot_sync(FULL, cand);
            if (cand) list[n + __popc(bal & ((1u << lane) - 1u))] = (uint16_t)i;
            n += __popc(bal);
        }
        __syncwarp();
        for (int i = n - 1; i >= 1; i--) {                            // Fisher-Yates from the top (legacy shuffle)
            const int j = (int)mt.interval((uint32_t)i, lane);
            if (lane == 0) { const uint16_t t = list[i]; list[i] = list[j]; list[j] = t; }
        }
        __syncwarp();
        const int pct = (int)mt.randint(op.lo, op.hi, lane);
        int take = (int)ceil((double)n * ((double)pct / 100.0));     // novelty_wrappers.py:881,1025,1139
        if (take > n) take = n;
        const int value = op.kind == NGW_RESET_ADDITEM ? op.a : op.b;
        for (int t = lane; t < take; t += 32) {                       // distinct cells: the first `take` in list order
            const int i = list[t];
            if (op.kind == NGW_RESET_FENCE) m[i] = (int8_t)(m[i] | 0x80);   // mark; fences go in afterwards
            else if (i != agent) m[i] = (int8_t)value;
        }
        __syncwarp();
        if (op.kind == NGW_RESET_FENCE) {                             // add_fence_around: the union does not depend on order
            for (int i = lane; i < cells; i += 32) {
                const int v = m[i];
                if (!(v & 0x80)) continue;
                const int r = i / ms, c = i - r * ms;
                for (int rr = r - 1; rr <= r + 1; rr++)
                    for (int cc = c - 1; cc <= c + 1; cc++)
                        if (rr >= 0 && rr < ms && cc >= 0 && cc < ms && m[rr * ms + cc] == 0 && rr * ms + cc != agent)
                            m[rr * ms + cc] = (int8_t)op.a;
            }
            __syncwarp();
            for (int i = lane; i < cells; i += 32) {
                const int v = m[i];
                if (v & 0x80) m[i] = (int8_t)(v & 0x7F);
            }
            __syncwarp();
        }
    }
    __syncwarp();
    if (lane == 0) *pos_io = mt.pos;
    return err;
}

}  // namespace ngw
