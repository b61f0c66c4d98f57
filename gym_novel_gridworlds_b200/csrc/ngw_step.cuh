// ngw_step.cuh — the hot kernel of libngw_b200.so: fused step + novelties + LidarInFront (+ rollout), sm_100a only.
//
// Data layout in HBM (struct of arrays, rows padded to a multiple of 32 envs so a tile of 32 envs is one contiguous,
// 128-byte aligned span in every array):
//     map   int8  [Np][ms*ms]      pose uchar4 [Np] (row, col, facing, selected)      inventory int32 [Np][Is]
//     cfg_id uint8 [Np]            episode u32 [Np]     ep_len i32 [Np]     error_flags u32 [Np]
//
// step_kernel: one CTA = one tile of 32 envs, one lane = one env.  The tile's grid rows and inventory rows are brought
// into shared memory with two TMA 1-D bulk copies (cp.async.bulk + mbarrier), warp 0 runs the flattened reference step
// on the rows, all warps cast the LidarInFront beams into an observation tile in shared memory, and the inventory tile
// and observation tile leave with two TMA bulk stores; pose / reward / done / step_cost / result are plain coalesced
// accesses.  Algorithmic bytes per env-step are in DESIGN.md.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include "ngw_device.cuh"

namespace ngw {

// ------------------------------------------------------------------ PTX helpers (TMA 1-D bulk copies, mbarrier)
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// L2 cache-hinted variants (createpolicy + .L2::cache_hint).  The kernels load the state tiles and store the observation
// tile evict_first: streaming data (each tile is read once and its observations written once per step) should not linger
// in L2 — measured on C2 9.15 -> 8.82 us/step, C3 29.3 -> 28.0, C5 278 -> 274 (hinting the inventory store as well: 9.0)
__device__ __forceinline__ uint64_t policy_evict_first() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ void bulk_g2s_hint(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar, uint64_t pol) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)), "l"(pol)
                 : "memory");
}
__device__ __forceinline__ void bulk_s2g_hint(void* dst_gmem, const void* src_smem, uint32_t bytes, uint64_t pol) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;" ::"l"(dst_gmem),
                 "r"(smem_u32(src_smem)), "r"(bytes), "l"(pol)
                 : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    // try_wait sleeps in hardware; the time bound turns a lost transaction into a trap instead of a hung GPU
    if (mbar_try_wait(bar, parity)) return;
    long long t0 = clock64();
    while (!mbar_try_wait(bar, parity))
        if (clock64() - t0 > 4000000000ll) __trap();
}
__device__ __forceinline__ void bulk_s2g(void* dst_gmem, const void* src_smem, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(smem_u32(src_smem)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ------------------------------------------------------------------ parameters
struct StepParams {
    const DevConfig* dcfgs;     // global-memory copy of the configs (cold paths, and the hot path when NC == 0)
    int8_t* map;
    uchar4* pose;
    int32_t* inv;
    const uint8_t* cfg_id;
    uint32_t* episode;
    int32_t* ep_len;
    uint32_t* err;
    const int32_t* actions;     // nullptr => observe only (no step, no outputs but obs)
    unsigned char* obs;         // nullptr => no observation; rows of obs_row_bytes bytes (layout obs_format)
    float* reward;
    uint8_t* done;
    float* cost;
    uint8_t* result;
    double* stats;              // [NGW_STAT_SLOTS][NGW_STAT_COUNT]
    long long env_begin, env_end;   // env range of this launch (env_begin multiple of 32)
    long long first_gid;
    unsigned long long seed;
    int ms, cells, inv_stride, obs_dim;
    int map_bytes, inv_bytes, obs_bytes;                 // bytes of one 32-env tile of each array
    int obs_row_bytes, obs_format;                       // observation row layout (NGW_OBS_I32 / NGW_OBS_U8 / NGW_OBS_HITS)
    int obs_srow;               // one-step kernel: row stride of the observation tile in SHARED memory: obs_row_bytes, or
                                // 16 bytes more when the row is a multiple of 8 words (64-word rows would put every
                                // lane's row on the same bank: C4 / C5 measured 64-71 % of their shared wavefronts as conflicts)
    // shared-memory carve-up (bytes from the start of dynamic shared memory), all multiples of 128
    int off_luts, off_scratch, off_policy, off_in, off_obs;   // rollout kernel (one tile per CTA)
    int off_groups, group_bytes;                         // one-step kernel: tile group k lives at off_groups + k * group_bytes
    int tiles_per_cta, g_shift, n_tiles;                 // one-step kernel: tile groups per CTA, log2(warps per tile), tiles
    int lidar_mode;             // 1: every config takes the line-gather path with one shared geometry (the common case)
    int early_state;            // 1: this handle's state is complete already, state loads may precede griddepcontrol.wait
    int concurrent;             // step1w_kernel: 1 = this launch is independent of its predecessor (another handle's step, proven
                                // adjacent in a stream capture, disjoint buffers): the tile warps do not wait for it, only the gate warp
    int auto_reset, max_episode_steps;
    int lidar_uniform;          // every config has the same beam tables (then config 0's are read, warp-uniformly)
    // K-step rollout (n_steps > 1 or random policy): the tile stays in shared memory across the steps
    int n_steps;                // steps per launch (1 for ngw_step)
    int random_policy;          // 1 => actions drawn on the device (Philox), `actions` is only a non-null marker
    long long act_stride;       // elements between consecutive steps in `actions` / `actions_out`
    unsigned long long policy_seed;
    int32_t* done_count;        // optional: episodes finished per env during the launch
    int32_t* actions_out;       // optional: actions taken
    const int32_t* policy_w;    // closed-loop linear policy: int32 [obs_dim][policy_actions] (nullptr = off)
    const int32_t* policy_b;    // int32 [policy_actions]
    int policy_actions;
    uint16_t* msg;              // optional: info['message'] codes (enum ngw_msg | arg << 5)
    int32_t* reset_list;        // single-step auto-reset: finished envs are queued here ...
    int32_t* reset_count;       // ... and regenerated by reset_list_kernel right after this launch
};

// Kernel argument block: the parameters plus up to NC configs INLINE, so that every config read in the hot path
// is a constant-bank operand (c[0x0][..]) instead of a global load.  NC == 0 falls back to global memory.
template <int NC>
struct StepArgs {
    StepParams p;
    DevConfig cfg[NC > 0 ? NC : 1];
    // the config of an env whose config id is cfg_i
    __device__ __forceinline__ const DevConfig& config(int cfg_i) const {
        return (NC == 1) ? cfg[0] : (NC > 1 ? cfg[cfg_i] : p.dcfgs[cfg_i]);
    }
};

#define NGW_STAT_SLOTS 512
#define NGW_SMEM_HDR 256            // mbarriers, zero pad, pose hand-over

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    return v;
}

// ------------------------------------------------------------------ tile plumbing shared by the step and rollout kernels
// Lidar tables read with per-lane indices, staged in shared memory: config 0's first-sample table, every inline config's
// item -> slot table (NC == 0: the lanes read both from the global config table instead).
template <int NC>
__device__ __forceinline__ void stage_lidar_luts(const StepArgs<NC>& args, uint8_t* sfirstk, int8_t* sslot) {
    if (NC > 0) {                                                     // config tables are kernel arguments (constant bank)
        if (threadIdx.x < NGW_MAX_MAP_SIZE / 4)
            reinterpret_cast<uint32_t*>(sfirstk)[threadIdx.x] =
                reinterpret_cast<const uint32_t*>(args.cfg[0].lidar.firstk)[threadIdx.x];
#pragma unroll
        for (int k = 0; k < NC; k++)
            if (threadIdx.x < NGW_MAX_ITEMS / 4)
                reinterpret_cast<uint32_t*>(sslot + k * NGW_MAX_ITEMS)[threadIdx.x] =
                    reinterpret_cast<const uint32_t*>(args.cfg[k].c.lidar_slot)[threadIdx.x];
    }
}

// the lane's lidar tables: the staged ones (stage_lidar_luts), or config cfg_i's in global memory when NC == 0
template <int NC>
__device__ __forceinline__ LidarLuts lane_luts(const StepParams& p, const uint8_t* sfirstk, const int8_t* sslot, int cfg_i) {
    LidarLuts luts;
    if (NC > 0) { luts.slot = sslot + cfg_i * NGW_MAX_ITEMS; luts.firstk = sfirstk; }
    else { luts.slot = p.dcfgs[cfg_i].c.lidar_slot; luts.firstk = p.dcfgs[cfg_i].lidar.firstk; }
    return luts;
}

// one thread: the tile's grid rows and inventory rows -> shared memory, completing on `bar`, L2 policy `pol`
__device__ __forceinline__ void issue_tile_loads(const StepParams& p, uint64_t* bar, int8_t* smap, const int8_t* gmap,
                                                 int32_t* sinv, const int32_t* ginv, uint64_t pol) {
    mbar_expect_tx(bar, (uint32_t)(p.map_bytes + p.inv_bytes));
    bulk_g2s_hint(smap, gmap, (uint32_t)p.map_bytes, bar, pol);
    bulk_g2s_hint(sinv, ginv, (uint32_t)p.inv_bytes, bar, pol);
}

// the action table entry of `action`; NGW_OP_INVALID for an id outside the config's actions
__device__ __forceinline__ ngw_action_entry decode_action(const ngw_config& cfg, int action) {
    ngw_action_entry a;
    a.op = NGW_OP_INVALID;
    if (action >= 0 && action < cfg.n_actions) {
        uint2 raw = *reinterpret_cast<const uint2*>(&cfg.actions[action]);
        memcpy(&a, &raw, sizeof(a));
    }
    return a;
}

// One-step kernels: episode bookkeeping after a valid step of env e — truncation at max_episode_steps (a harness knob: it
// sets o.done), the episode length, and whether the env is reset.  ld.cg: another grid may overlap this one.  (The
// rollouts keep this inline with a plain load: there ep_len is read once per step on the step's dependent chain, and
// ld.cg measured 1.6 % fewer env-steps/s on the C2 rollout, B200 at 1000 W.)
__device__ __forceinline__ int end_of_step(const StepParams& p, long long e, StepOut& o) {
    int finished = o.done;
    if (p.max_episode_steps > 0) {
        int len = __ldcg(&p.ep_len[e]) + 1;
        if (len >= p.max_episode_steps) { finished = 1; o.done = 1; }
        p.ep_len[e] = finished && p.auto_reset ? 0 : len;
    }
    return finished && p.auto_reset;
}

// whole warp: append the lanes with did_reset to the auto-reset queue that reset_list_kernel consumes
__device__ __forceinline__ void queue_resets(const StepParams& p, int lane, long long e, int did_reset) {
    const uint32_t bal = __ballot_sync(0xFFFFFFFFu, did_reset);
    if (bal != 0) {
        int base = 0;
        if (lane == 0) base = atomicAdd(p.reset_count, __popc(bal));
        base = __shfl_sync(0xFFFFFFFFu, base, 0);
        if (did_reset) p.reset_list[base + __popc(bal & ((1u << lane) - 1u))] = (int)e;
    }
}

// one thread: add one set of episode statistics into statistics slot `slot` (mod NGW_STAT_SLOTS)
__device__ __forceinline__ void flush_stats(double* stats, unsigned slot, int steps, int reward, float cost, int done,
                                            int succ, int reset, int invalid) {
    double* s = stats + (size_t)(slot % NGW_STAT_SLOTS) * NGW_STAT_COUNT;
    atomicAdd(&s[NGW_STAT_STEPS], (double)steps);
    atomicAdd(&s[NGW_STAT_REWARD_SUM], (double)reward);
    atomicAdd(&s[NGW_STAT_COST_SUM], (double)cost);
    if (done) atomicAdd(&s[NGW_STAT_EPISODES], (double)done);
    if (succ) atomicAdd(&s[NGW_STAT_SUCCESSES], (double)succ);
    if (reset) atomicAdd(&s[NGW_STAT_RESETS], (double)reset);
    if (invalid) atomicAdd(&s[NGW_STAT_INVALID], (double)invalid);
}

// threads t, t + nt, ...: copy `bytes` (a multiple of 16) in 16-byte words
__device__ __forceinline__ void copy16(void* dst, const void* src, int bytes, int t, int nt) {
    const uint4* s4 = reinterpret_cast<const uint4*>(src);
    uint4* d4 = reinterpret_cast<uint4*>(dst);
    for (int i = t; i < (bytes >> 4); i += nt) d4[i] = s4[i];
}

// threads t, t + nt, ...: the valid rows of a partial observation tile -> HBM (srow: the row stride in shared memory)
__device__ __forceinline__ void copy_obs_rows(const StepParams& p, long long e0, const unsigned char* sobs, int srow, int t,
                                              int nt) {
    const int rows = (int)(p.env_end - e0 < 32 ? p.env_end - e0 : 32), words = p.obs_row_bytes >> 2;
    for (int r = 0; r < rows; r++) {
        uint32_t* grow = reinterpret_cast<uint32_t*>(p.obs + (e0 + r) * p.obs_row_bytes);
        const uint32_t* srow_p = reinterpret_cast<const uint32_t*>(sobs + r * srow);
        for (int i = t; i < words; i += nt) grow[i] = srow_p[i];
    }
}

// zero the shared memory [a, end) (shared-memory addresses), 16 bytes per thread and pass, `step` bytes apart
__device__ __forceinline__ void zero_span(uint32_t a, uint32_t end, uint32_t step) {
#pragma unroll 4
    for (; a < end; a += step) asm volatile("st.shared.v4.b32 [%0], {%1, %1, %1, %1};" ::"r"(a), "r"(0) : "memory");
}

// one warp: a full observation tile -> HBM (L2 policy `pol`), one bulk store when the tile's rows are contiguous in shared
// memory, else one per row (lane l stores row l)
__device__ __forceinline__ void store_obs_tile(const StepParams& p, long long e0, const unsigned char* sobs, int lane,
                                               uint64_t pol) {
    unsigned char* gobs = p.obs + e0 * p.obs_row_bytes;
    if (p.obs_srow == p.obs_row_bytes) {
        if (lane == 0) bulk_s2g_hint(gobs, sobs, (uint32_t)p.obs_bytes, pol);
    } else {
        bulk_s2g_hint(gobs + lane * p.obs_row_bytes, sobs + lane * p.obs_srow, (uint32_t)p.obs_row_bytes, pol);
    }
}

// Cold: fused auto-reset.  Called by the whole step warp; every lane that finished an episode is regenerated in turn by
// all 32 lanes (reset_env_warp), then its grid row goes back to HBM with coalesced stores.
static __device__ __noinline__ void auto_reset_warp(const StepParams& p, const DevConfig* dcfgs, int cfg_i, bool need,
                                             int8_t* smap, int32_t* sinv, uint32_t* hist, long long e0, uchar4& ps) {
    const int lane = threadIdx.x & 31;
    __syncwarp();                                                    // every lane's step writes to the tile are visible
    uint32_t pending = __ballot_sync(0xFFFFFFFFu, need);
    while (pending) {
        const int src = __ffs(pending) - 1;
        pending &= pending - 1;
        const long long e = e0 + src;
        const int ci = __shfl_sync(0xFFFFFFFFu, cfg_i, src);
        uint32_t ep = p.episode[e] + 1;
        __syncwarp();
        if (lane == 0) p.episode[e] = ep;
        int8_t* m = smap + src * p.cells;
        int32_t* inv = sinv + src * p.inv_stride;
        int r = 0, c = 0, f = 0, sel = 0;
        uint32_t err = reset_env_warp(&dcfgs[ci].c, m, inv, p.ms, p.inv_stride, p.seed, (uint64_t)(p.first_gid + e), ep,
                                      true, 0, NGW_MAX_RESET_OPS, hist, r, c, f, sel);
        int8_t* grow = p.map + e * p.cells;
        for (int i = lane; i < p.cells; i += 32) grow[i] = m[i];
        if (lane == src) {
            ps = make_uchar4((unsigned char)r, (unsigned char)c, (unsigned char)f, (unsigned char)sel);
            if (err) p.err[e] |= err;
        }
        __syncwarp();
    }
}

// Episode statistics of one tile: warp reductions + one atomic per counter into one of NGW_STAT_SLOTS slots.
__device__ __forceinline__ void tile_stats(double* stats, unsigned slot, int lane, int valid, int done, int success, int did_reset,
                                           int invalid, int reward, float cost) {
    // five small counts (each <= 32) share one reduction: 6 bits apiece
    unsigned packed = (unsigned)(valid ? done : 0) | ((unsigned)success << 6) | ((unsigned)did_reset << 12) |
                      ((unsigned)invalid << 18) | ((unsigned)(valid ? 1 : 0) << 24);
    packed = __reduce_add_sync(0xFFFFFFFFu, packed);
    const int r_sum = __reduce_add_sync(0xFFFFFFFFu, reward);
    const float c_sum = warp_sum(cost);
    if (lane == 0) {
        const int n_done = packed & 63, n_succ = (packed >> 6) & 63, n_reset = (packed >> 12) & 63;
        const int n_inv = (packed >> 18) & 63, n_valid = (packed >> 24) & 63;
        flush_stats(stats, slot, n_valid - n_inv, r_sum, c_sum, n_done, n_succ, n_reset, n_inv);
    }
}

// ------------------------------------------------------------------ the K-STEP ROLLOUT kernel (ngw_rollout, ngw_rollout_policy)
// SURVEY §8f N1.  One CTA = one tile of 32 consecutive envs that stays in shared memory for n_steps steps; lane l owns env
// l.  Warp 0 runs the steps; actions come from a [K][N] tensor (next step's action prefetched behind the current step),
// from an on-device uniform random policy (Philox keyed by global env id and step), or — the closed loop — from an integer
// linear policy evaluated on each step's LidarInFront observation.  The closed loop never materialises that observation:
// the lidar feeds a PolicySink that accumulates  score[a] = bias[a] + sum_j obs[j] W[j][a]  hit by hit, with W staged in
// shared memory.  Finished lanes are regenerated in place by the step warp (auto_reset_warp).  After the last step all G
// warps cast the final observation, which leaves with the inventory tile through two TMA bulk stores; the other outputs are
// per-env sums (reward, step_cost, episodes finished) and the last step's done / result.
#define NGW_CLASS1_OPS ((1u << NGW_OP_FORWARD) | (1u << NGW_OP_BREAK) | (1u << NGW_OP_PLACE_TREE_TAP) | \
                        (1u << NGW_OP_EXTRACT_RUBBER) | (1u << NGW_OP_EXTRACT_STRING) | (1u << NGW_OP_CHOP) | (1u << NGW_OP_JUMP))

template <int NC>
__global__ void __launch_bounds__(256) rollout_kernel(const __grid_constant__ StepArgs<NC> args) {
    extern __shared__ __align__(128) unsigned char smem[];
    const StepParams& p = args.p;
    const int lane = threadIdx.x & 31, g = threadIdx.x >> 5, G = blockDim.x >> 5;
    const long long e0 = p.env_begin + (long long)blockIdx.x * 32;
    const long long e = e0 + lane;
    const bool valid = e < p.env_end;
    const bool full_tile = e0 + 32 <= p.env_end;

    uint64_t* bar = reinterpret_cast<uint64_t*>(smem);               // "tile landed" barrier
    int8_t* szero = reinterpret_cast<int8_t*>(smem + 32);            // 8 bytes that always read 0 (landed lidar beams park here)
    uchar4* spose = reinterpret_cast<uchar4*>(smem + 64);            // pose after the last step, for the other warps
    uint8_t* sfirstk = smem + p.off_luts;                            // lidar tables read with per-lane indices
    int8_t* sslot = reinterpret_cast<int8_t*>(smem + p.off_luts + NGW_MAX_MAP_SIZE);
    uint32_t* sscratch = reinterpret_cast<uint32_t*>(smem + p.off_scratch);   // radix-select scratch of the in-place auto-reset
    int32_t* spol = reinterpret_cast<int32_t*>(smem + p.off_policy); // closed loop: bias [16] | W [obs_dim][A]
    int8_t* smap = reinterpret_cast<int8_t*>(smem + p.off_in);
    int32_t* sinv = reinterpret_cast<int32_t*>(smem + p.off_in + p.map_bytes);
    unsigned char* sobs = smem + p.off_obs;
    const bool closed_loop = p.policy_w != nullptr;

    // ---- prologue without global state: barrier, zero pad, lidar tables, zeroed observation tile
    const int8_t* gmap = p.map + e0 * p.cells;
    int32_t* ginv = p.inv + e0 * p.inv_stride;
    if (threadIdx.x == 0) {
        mbar_init(bar, 1);
        *reinterpret_cast<uint64_t*>(szero) = 0ull;
    }
    stage_lidar_luts<NC>(args, sfirstk, sslot);
    if (p.obs != nullptr) {
        const uint4 z = make_uint4(0, 0, 0, 0);
        uint4* o4 = reinterpret_cast<uint4*>(sobs);
        for (int i = threadIdx.x; i < (p.obs_bytes >> 4); i += blockDim.x) o4[i] = z;
    }
    __syncthreads();                                                 // barrier init visible before anyone waits on it
    asm volatile("griddepcontrol.wait;" ::: "memory");               // previous kernel of the stream done + visible

    // ---- stage the tile: grid rows + inventory rows (state arrays are padded, a full tile is always readable)
    if (threadIdx.x == 0) issue_tile_loads(p, bar, smap, gmap, sinv, ginv, policy_evict_first());
    if (closed_loop) {                                               // the policy's weights, once per CTA
        const int n_w = p.obs_dim * p.policy_actions;
        for (int i = threadIdx.x; i < 16; i += blockDim.x) spol[i] = i < p.policy_actions ? p.policy_b[i] : 0;
        for (int i = threadIdx.x; i < n_w; i += blockDim.x) spol[16 + i] = p.policy_w[i];
    }

    // ---- while the copies fly: per-lane scalars
    const int cfg_i = (NC == 1) ? 0 : (int)p.cfg_id[e];
    const DevConfig& dc = args.config(cfg_i);
    const ngw_config& cfg = dc.c;
    const LidarDev& beam_tables = (NC > 1 && p.lidar_uniform) ? args.cfg[0].lidar : dc.lidar;
    LidarLuts luts = lane_luts<NC>(p, sfirstk, sslot, cfg_i);
    if (NC > 1 && !p.lidar_uniform) luts.slot = nullptr;              // heterogeneous beam tables: pointer-walking path
    ObsRow orow;
    orow.p = sobs + lane * p.obs_row_bytes;
    orow.fmt = p.obs_format;
    uchar4 ps = make_uchar4(0, 0, 0, 0);
    int action = 0;
    const bool given_actions = !(p.random_policy || closed_loop);     // else `actions` is only a non-null marker
    if (g == 0) {
        ps = p.pose[e];
        if (valid && given_actions) action = p.actions[e];
    }

    mbar_wait(bar, 0);
    __syncthreads();                                                 // policy weights visible to the step warp

    EnvRow env;
    env.m = smap + lane * p.cells;
    env.gm = p.map + e * p.cells;
    env.inv = sinv + lane * p.inv_stride;
    env.ms = p.ms;

    if (g == 0) {
        env.set_pose(ps);
        StepOut o;
        o.clear();
        float reward_sum = 0.0f, cost_sum = 0.0f;
        int done_count = 0;
        // the sink needs the line-gather lidar (lidar_observe would take the same branch); otherwise the observation row
        // is materialised and scanned
        const bool use_sink = closed_loop && dc.lidar.lines && luts.slot != nullptr && (p.ms <= 32 || !dc.lidar.fast);
        RandomPolicy rpol;
        rpol.first = 0u; rpol.w[0] = rpol.w[1] = rpol.w[2] = rpol.w[3] = 0u;
        for (int t = 0; t < p.n_steps; t++) {
            int next_action = 0;                                      // prefetch the next step's action behind this step
            if (given_actions && t + 1 < p.n_steps && valid) next_action = p.actions[(t + 1) * p.act_stride + e];
            if (closed_loop) {                                        // observe, then greedy linear policy (int32 arithmetic)
                const int n_valid = cfg.n_actions < p.policy_actions ? cfg.n_actions : p.policy_actions;
                if (use_sink) {
                    PolicySink sink;
                    sink.init(spol + 16, spol, p.policy_actions);
                    if (valid && cfg.n_beams > 0) {
                        lidar_lines<false, PolicySink>(env, cfg, beam_tables, luts, sink, 0xF);
                        obs_tail<PolicySink>(env, cfg, sink, dc.lidar.tail_first);
                    }
                    action = sink.argmax(n_valid);
                } else {
                    int32_t* row = reinterpret_cast<int32_t*>(orow.p);
                    for (int j = 0; j < p.obs_dim; j++) row[j] = 0;
                    if (valid && cfg.n_beams > 0) lidar_observe<false>(env, dc, beam_tables, luts, orow, szero, 0, 1, true);
                    PolicySink sink;
                    sink.init(spol + 16, spol, p.policy_actions);
                    const int D = cfg.n_lidar_items * cfg.n_beams + cfg.n_inv_obs;
                    for (int j = 0; j < D; j++) {
                        const int v = row[j];
                        if (v != 0) sink.add(j, v);                    // the observation is sparse (<= 8 hits + inventory)
                    }
                    action = sink.argmax(n_valid);
                }
            } else if (p.random_policy && valid) {                    // uniform over the config's action ids
                action = rpol.draw(p.policy_seed, (uint64_t)(p.first_gid + e), (uint32_t)t, (uint32_t)(cfg.n_actions > 0 ? cfg.n_actions : 1));
            }
            if (p.actions_out != nullptr && valid) p.actions_out[t * p.act_stride + e] = action;
            o.clear();
            int invalid = 0, did_reset = 0, success = 0;
            if (valid) {
                const ngw_action_entry a = decode_action(cfg, action);
                if (a.op == NGW_OP_INVALID) {                         // wrappers.py:76 / pogostick_v1_env.py:236 would raise
                    invalid = 1;
                    p.err[e] |= NGW_ERR_INVALID_ACTION;
                } else {
                    step_env(env, cfg, a, o);
                    success = o.goal;
                    int finished = o.done;
                    if (p.max_episode_steps > 0) {
                        int len = p.ep_len[e] + 1;
                        if (len >= p.max_episode_steps) { finished = 1; o.done = 1; }   // harness truncation knob
                        p.ep_len[e] = finished && p.auto_reset ? 0 : len;
                    }
                    if (finished && p.auto_reset) did_reset = 1;
                }
                ps = env.pose();
                reward_sum += (float)o.reward; cost_sum += o.cost; done_count += o.done;
            }
            if (p.auto_reset) {
                // the next step needs the new episode now -> regenerate in place, warp-cooperatively
                if (__ballot_sync(0xFFFFFFFFu, did_reset) != 0) {
                    auto_reset_warp(p, p.dcfgs, cfg_i, did_reset != 0, smap, sinv, sscratch, e0, ps);
                    env.set_pose(ps);
                }
            }
            tile_stats(p.stats, blockIdx.x, lane, valid, o.done, success, did_reset, invalid, o.reward, o.cost);
            action = next_action;
        }
        if (closed_loop && !use_sink) {                               // the last policy observation must not leak into the final one
            int32_t* row = reinterpret_cast<int32_t*>(orow.p);
            for (int j = 0; j < p.obs_dim; j++) row[j] = 0;
        }
        if (valid) {
            p.pose[e] = ps;
            p.reward[e] = reward_sum;
            p.done[e] = (uint8_t)o.done;
            p.cost[e] = cost_sum;
            p.result[e] = (uint8_t)o.result;
            if (p.done_count != nullptr) p.done_count[e] = done_count;
            if (p.msg != nullptr) p.msg[e] = (uint16_t)o.msg;
        }
        if (G > 1) spose[lane] = ps;
    }
    if (G > 1) {
        __syncthreads();                                             // step results (grid, inventory, pose) visible to all warps
        ps = spose[lane];
        env.set_pose(ps);
    }

    // ---- LidarInFront observation of the final state into the shared-memory tile
    if (p.obs != nullptr && valid && cfg.n_beams > 0)
        lidar_observe<false>(env, dc, beam_tables, luts, orow, szero, g, G, g == G - 1);

    // ---- write back: inventory tile and observation tile.  Every thread orders its generic-proxy writes to the tiles
    //      before the async proxy reads them (fence before the barrier), then one thread issues.
    fence_async_smem();
    __syncthreads();
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (full_tile) {
        if (threadIdx.x == 0) {
            bulk_s2g(ginv, sinv, (uint32_t)p.inv_bytes);
            if (p.obs != nullptr)
                bulk_s2g_hint(p.obs + e0 * p.obs_row_bytes, sobs, (uint32_t)p.obs_bytes, policy_evict_first());
            bulk_commit();
            bulk_wait_read<0>();                                     // shared memory must outlive the bulk stores' reads
        }
    } else {
        copy16(ginv, sinv, p.inv_bytes, threadIdx.x, blockDim.x);
        if (p.obs != nullptr) copy_obs_rows(p, e0, sobs, p.obs_row_bytes, threadIdx.x, blockDim.x);
    }
}

// ------------------------------------------------------------------ the ONE-STEP kernel (ngw_step / ngw_observe)
// The hot kernel.  One CTA = tiles_per_cta TILE GROUPS that run concurrently and independently; a tile group = G warps
// (1, 2 or 4) working on one tile of 32 consecutive envs, lane l of every warp owning env l.  Per group:
//   prologue   mbarrier init, zeroed observation tile (no global state is touched before griddepcontrol.wait)
//   load       two TMA bulk copies bring the tile's grid rows and inventory rows into shared memory
//   step       split by ACTION CLASS over the first two warps: warp 0 executes the lanes whose action is a turn / craft /
//              select, warp 1 the lanes that move or touch the block in front — each walks half of the divergent paths
//   lidar      after one group barrier all G warps cast the LidarInFront lines of their lane's env (G = 2: axis / diagonals)
//   store      two TMA bulk stores (inventory tile, observation tile), then warp 0 writes the per-env outputs of ALL lanes
//              (handed over through shared memory, so the stores are full 128-byte lines) and folds the statistics
// Several groups per CTA exist because an empty launch of one-tile CTAs already costs 3.4 us on C2 (2048 CTA launches of
// 64 threads); with 7 groups per CTA the same tiles are 293 CTAs.  Groups synchronise with their own named barrier
// (bar.sync 1 + group), never with the whole CTA after the prologue.
struct TileOut {            // per-env hand-over from the warp that stepped the lane: 16 bytes
    uchar4 ps;              // pose after the step
    uint32_t bits;          // reward (int16) | done << 16 | result << 17 | success << 18 | reset << 19 | invalid << 20 | stepped << 21
    float cost;
    uint32_t msg;
};
#define NGW_GROUP_HDR 640   // mbarrier (8) | zero pad (8) | .. | TileOut[32] at +64 | pad to a multiple of 128
#define NGW_CTA_HDR 128     // per-CTA statistics accumulators

// kOne: the CTA is a single tile group, which synchronises on barrier 0 — a register-indexed bar.sync makes ptxas
// reserve all 16 named barriers, and 64 / 16 = 4 such CTAs per SM is too few when every CTA is one tile.
template <bool kOne>
__device__ __forceinline__ void group_sync(int grp, int G) {
    if (G == 1) __syncwarp();
    else if (kOne) __syncthreads();
    else asm volatile("bar.sync %0, %1;" ::"r"(grp + 1), "r"(G * 32) : "memory");
}

// kAlias (one tile per CTA only): the observation tile ALIASES the grid / inventory rows, as in step1w_kernel — the lidar
// hits and the inventory tail wait in registers (RegSink) until the rows have been consumed.  A 40x40 tile is then 52 KB
// instead of 61 KB: four tiles per SM instead of three (C5).
template <int NC, bool kOne, bool kAlias = false>
__global__ void __launch_bounds__(512) step1_kernel(const __grid_constant__ StepArgs<NC> args) {
    extern __shared__ __align__(128) unsigned char smem[];
    const StepParams& p = args.p;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int G = 1 << p.g_shift;
    const int grp = wid >> p.g_shift, g = wid & (G - 1);
    const int gt = threadIdx.x & (32 * G - 1);                        // thread index inside the tile group
    // concurrent mode (see step1w_kernel): block 0 is the GATE — it waits for the preceding grid and only then lets the
    // next launch start; the tile CTAs never wait
    if (p.concurrent && blockIdx.x == 0) {
        asm volatile("griddepcontrol.wait;" ::: "memory");
        asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
        return;
    }
    const int tile = ((int)blockIdx.x - p.concurrent) * p.tiles_per_cta + grp;
    const bool active = tile < p.n_tiles;
    const long long e0 = p.env_begin + (long long)tile * 32;
    const long long e = e0 + lane;
    const bool valid = active && e < p.env_end;
    const bool full_tile = e0 + 32 <= p.env_end;
    const bool stepping = p.actions != nullptr;

    int* scta = reinterpret_cast<int*>(smem);                         // [0] counts a, [1] counts b, [2] reward, [3] cost (float), [4] groups done
    uint8_t* sfirstk = smem + p.off_luts;                             // lidar tables read with per-lane indices
    int8_t* sslot = reinterpret_cast<int8_t*>(smem + p.off_luts + NGW_MAX_MAP_SIZE);
    unsigned char* gbase = smem + p.off_groups + grp * p.group_bytes;
    uint64_t* bar = reinterpret_cast<uint64_t*>(gbase);               // "tile landed" barrier
    int8_t* szero = reinterpret_cast<int8_t*>(gbase + 8);             // 8 bytes that always read 0 (landed lidar beams park here)
    TileOut* sout = reinterpret_cast<TileOut*>(gbase + 64);
    int8_t* smap = reinterpret_cast<int8_t*>(gbase + NGW_GROUP_HDR);
    int32_t* sinv = reinterpret_cast<int32_t*>(gbase + NGW_GROUP_HDR + p.map_bytes);
    unsigned char* sobs = gbase + NGW_GROUP_HDR + (kAlias ? 0 : p.map_bytes + p.inv_bytes);
    const uint32_t in_bytes = (uint32_t)(p.map_bytes + p.inv_bytes);

    // ---- prologue without global state: barriers, zero pad, lidar tables
    if (threadIdx.x < 8) scta[threadIdx.x] = 0;
    if (gt == 0) {
        mbar_init(bar, 1);
        *reinterpret_cast<uint64_t*>(szero) = 0ull;
    }
    stage_lidar_luts<NC>(args, sfirstk, sslot);
    __syncthreads();                                                  // the only CTA-wide barrier

    // ---- stage the tile: grid rows + inventory rows (state arrays are padded, a full tile is always readable).
    // p.early_state: the launch that precedes this one in the stream does not belong to this handle, so this handle's
    // state was last written at least two launches back and is complete and visible already (the predecessor passed its
    // own griddepcontrol.wait before it let this launch start): the state loads go out BEFORE the wait and overlap the
    // predecessor's tail.  Otherwise they follow the wait.
    const int8_t* gmap = p.map + e0 * p.cells;
    int32_t* ginv = p.inv + e0 * p.inv_stride;
    const uint64_t pol_first = policy_evict_first();
    auto issue_loads = [&]() {
        if (gt == 0) issue_tile_loads(p, bar, smap, gmap, sinv, ginv, pol_first);
    };
    const int n_cls = G >= 2 ? 2 : 1;                                 // warps that take part in the step
    uchar4 ps = make_uchar4(0, 0, 0, 0);
    const bool early = p.early_state && active;
    if (early) {
        issue_loads();
        if (g < n_cls) ps = __ldcg(&p.pose[e]);
    }
    if (p.obs != nullptr)                                             // the group zeroes its observation tile while the loads fly
        zero_span(smem_u32(sobs) + (uint32_t)gt * 16u + (kAlias ? in_bytes : 0u),   // (alias: only the part beyond the rows)
                  smem_u32(sobs) + 32u * (uint32_t)p.obs_srow, 512u * (uint32_t)G);
    if (!p.concurrent) {
        asm volatile("griddepcontrol.wait;" ::: "memory");            // previous kernel of the stream done + visible
        // trigger right after the wait (rather than once the stores are issued): C2 7.70 -> 7.60 us/step
        asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    }
    if (!active) { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); return; }
    if (!early) issue_loads();

    // ---- while the copies fly: per-lane scalars
    const int cfg_i = (NC == 1) ? 0 : (int)__ldcg(&p.cfg_id[e]);
    const DevConfig& dc = args.config(cfg_i);
    const ngw_config& cfg = dc.c;
    int action = 0;
    if (g < n_cls) {
        if (!early) ps = __ldcg(&p.pose[e]);
        if (stepping && valid) action = __ldcg(&p.actions[e]);
    }

    mbar_wait(bar, 0);

    EnvRow env;
    env.m = smap + lane * p.cells;
    env.gm = p.map + e * p.cells;
    env.inv = sinv + lane * p.inv_stride;
    env.ms = p.ms;

    if (g < n_cls) {
        env.set_pose(ps);
        bool mine = !stepping && g == 0;                              // this warp publishes this lane's hand-over record
        uint32_t bits = 0;
        StepOut o;
        o.clear();
        if (stepping) {
            // (decode_action plus the lane's validity: calling it with an id of -1 for past-the-end lanes costs
            // step1_kernel<1, true, true> a register)
            ngw_action_entry a;
            a.op = NGW_OP_INVALID;
            if (valid && action >= 0 && action < cfg.n_actions) {
                uint2 raw = *reinterpret_cast<const uint2*>(&cfg.actions[action]);
                memcpy(&a, &raw, sizeof(a));
            }
            // action class of the lane: which of the stepping warps executes it (lanes past the batch end: warp 0)
            mine = n_cls == 1 || (int)((NGW_CLASS1_OPS >> a.op) & 1u) == g;
            int did_reset = 0;
            if (mine && valid) {
                bits = 1u << 21;
                if (a.op == NGW_OP_INVALID) {                         // wrappers.py:76 / pogostick_v1_env.py:236 would raise
                    bits |= 1u << 20;
                    atomicOr(&p.err[e], NGW_ERR_INVALID_ACTION);
                } else {
                    step_env(env, cfg, a, o);
                    if (o.goal) bits |= 1u << 18;
                    did_reset = end_of_step(p, e, o);
                    if (did_reset) bits |= 1u << 19;
                }
                ps = env.pose();
                bits |= ((uint32_t)o.reward & 0xFFFFu) | ((uint32_t)o.done << 16) | ((uint32_t)o.result << 17);
            }
            // queue the finished envs; reset_list_kernel (next in the stream, one warp per env at full occupancy)
            // regenerates them and overwrites their observation rows
            if (p.auto_reset) queue_resets(p, lane, e, did_reset);
        }
        if (mine) {                                                   // one 16-byte record per lane, written by its stepping warp
            TileOut t;
            t.ps = ps; t.bits = bits; t.cost = o.cost; t.msg = (uint32_t)o.msg;
            *reinterpret_cast<uint4*>(&sout[lane]) = *reinterpret_cast<uint4*>(&t);
        }
    }
    group_sync<kOne>(grp, G);                                               // step results (grid, inventory, hand-over) visible to the group
    ps = sout[lane].ps;
    env.set_pose(ps);
    if (kAlias && stepping) {                                         // the inventory tile leaves before its rows are overwritten
        if (full_tile) {
            fence_async_smem();
            group_sync<kOne>(grp, G);
            if (gt == 0) { bulk_s2g(ginv, sinv, (uint32_t)p.inv_bytes); bulk_commit(); }
        } else {
            copy16(ginv, sinv, p.inv_bytes, gt, 32 * G);
        }
    }

    // ---- LidarInFront observation of the new state into the shared-memory tile
    if (kAlias) {
        if (p.obs != nullptr) {
            RegSink<NGW_REGSINK_TAIL> sink;
            sink.init(p.obs_format);
            const bool look = valid && cfg.n_beams > 0;
            if (look) {
                LidarLuts luts = lane_luts<NC>(p, sfirstk, sslot, cfg_i);
                if (NC > 1 && !p.lidar_uniform) luts.slot = nullptr;
                lidar_observe<false, RegSink<NGW_REGSINK_TAIL> >(env, dc, (NC > 1 && p.lidar_uniform) ? args.cfg[0].lidar : dc.lidar,
                                                                 luts, sink, szero, g, G, g == G - 1);
            }
            if (gt == 0) bulk_wait_read<0>();                         // the inventory store has read its rows
            group_sync<kOne>(grp, G);                                 // ... and every warp is done with the grid rows
            zero_span(smem_u32(sobs) + (uint32_t)gt * 16u, smem_u32(sobs) + min(in_bytes, 32u * (uint32_t)p.obs_srow),
                      512u * (uint32_t)G);
            group_sync<kOne>(grp, G);
            if (look) {
                sink.flush(smem_u32(sobs) + (uint32_t)(lane * p.obs_srow), smem_u32(gbase + 16), cfg.n_lidar_items,
                           obs_tail_offset(p.obs_format, cfg.n_lidar_items, cfg.n_beams), g == G - 1 ? cfg.n_inv_obs : 0);
            }
        }
    } else
    if (p.obs != nullptr && valid && cfg.n_beams > 0) {
        ObsRow orow;
        orow.p = sobs + lane * p.obs_srow;
        orow.fmt = p.obs_format;
        LidarLuts luts = lane_luts<NC>(p, sfirstk, sslot, cfg_i);
        if (p.lidar_mode == 1) {                                      // every config: line gather, one shared geometry
            const int sel = lidar_line_share(g, G);
            if (sel) lidar_lines<false, ObsRow>(env, cfg, (NC > 0) ? args.cfg[0].lidar : dc.lidar, luts, orow, sel);
            if (g == G - 1) obs_tail<ObsRow>(env, cfg, orow, dc.lidar.tail_first);
        } else {
            if (NC > 1 && !p.lidar_uniform) luts.slot = nullptr;      // heterogeneous beam tables: pointer-walking path
            lidar_observe<false>(env, dc, (NC > 1 && p.lidar_uniform) ? args.cfg[0].lidar : dc.lidar, luts, orow, szero,
                                 g, G, g == G - 1);
        }
    }

    // ---- write back: inventory tile (only when stepping) and observation tile.  Every thread orders its generic-proxy
    //      writes to the tiles before the async proxy reads them (fence before the barrier), then one thread issues.
    fence_async_smem();
    group_sync<kOne>(grp, G);
    if (full_tile) {
        if (!kAlias && gt == 0 && stepping) bulk_s2g(ginv, sinv, (uint32_t)p.inv_bytes);
        if (p.obs != nullptr && g == 0) store_obs_tile(p, e0, sobs, lane, pol_first);
        if (g == 0) bulk_commit();
    } else {
        if (stepping && !kAlias) copy16(ginv, sinv, p.inv_bytes, gt, 32 * G);
        if (p.obs != nullptr) copy_obs_rows(p, e0, sobs, p.obs_srow, gt, 32 * G);
    }

    // ---- per-env outputs (full lines, one warp) and episode statistics, behind the tile stores
    if (g == 0 && stepping) {
        const uint4 raw = *reinterpret_cast<const uint4*>(&sout[lane]);
        const uint32_t bits = raw.y;
        const int reward = (int)(short)(bits & 0xFFFFu);
        const float cost = __uint_as_float(raw.z);
        if (valid) {
            p.pose[e] = *reinterpret_cast<const uchar4*>(&raw.x);
            p.reward[e] = (float)reward;
            p.done[e] = (uint8_t)((bits >> 16) & 1u);
            p.cost[e] = cost;
            p.result[e] = (uint8_t)((bits >> 17) & 1u);
            if (p.msg != nullptr) p.msg[e] = (uint16_t)raw.w;
        }
        // warp reductions, then shared-memory accumulators of the CTA; the last group to arrive flushes them with one
        // set of global atomics per CTA
        const uint32_t stepped = valid ? (bits >> 21) & 1u : 0u;
        const uint32_t a_cnt = stepped | ((valid ? (bits >> 16) & 1u : 0u) << 10) | (((bits >> 18) & 1u) << 20);     // steps | episodes | successes
        const uint32_t b_cnt = ((bits >> 19) & 1u) | (((bits >> 20) & 1u) << 10);                                       // resets | invalid
        const uint32_t a_sum = __reduce_add_sync(0xFFFFFFFFu, valid ? a_cnt : 0u);
        const uint32_t b_sum = __reduce_add_sync(0xFFFFFFFFu, valid ? b_cnt : 0u);
        const int r_sum = __reduce_add_sync(0xFFFFFFFFu, valid ? reward : 0);
        const float c_sum = warp_sum(valid ? cost : 0.0f);
        if (lane == 0) {
            int a_tot = (int)a_sum, b_tot = (int)b_sum, r_tot = r_sum;
            float c_tot = c_sum;
            bool flush = true;
            if (!kOne) {                                          // several groups: fold in shared memory, the last one flushes
                atomicAdd(&scta[0], a_tot);
                atomicAdd(&scta[1], b_tot);
                atomicAdd(&scta[2], r_tot);
                atomicAdd(reinterpret_cast<float*>(&scta[3]), c_tot);
                __threadfence_block();
                const int n_groups = min(p.tiles_per_cta, p.n_tiles - ((int)blockIdx.x - p.concurrent) * p.tiles_per_cta);
                flush = atomicAdd(&scta[4], 1) == n_groups - 1;
                if (flush) {
                    __threadfence_block();
                    a_tot = *reinterpret_cast<volatile int*>(&scta[0]); b_tot = *reinterpret_cast<volatile int*>(&scta[1]);
                    r_tot = *reinterpret_cast<volatile int*>(&scta[2]);
                    c_tot = *reinterpret_cast<volatile float*>(&scta[3]);
                }
            }
            if (flush) {
                const int n_step = a_tot & 1023, n_done = (a_tot >> 10) & 1023, n_succ = (a_tot >> 20) & 1023;
                const int n_reset = b_tot & 1023, n_inv = (b_tot >> 10) & 1023;
                flush_stats(p.stats, blockIdx.x, n_step - n_inv, r_tot, c_tot, n_done, n_succ, n_reset, n_inv);
            }
        }
    }

    // Programmatic dependent launch: this group's work is issued; once every group of the CTA got here the next kernel of
    // the stream may start scheduling its CTAs (its prologue touches no global state: it overlaps this kernel's stores).
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (g == 0) bulk_wait_read<0>();                                  // shared memory must outlive the bulk stores' reads
}

// ------------------------------------------------------------------ the ONE-STEP kernel, WARP-PER-TILE shape (one-wave launches)
// One warp owns one tile of 32 envs from load to store; a CTA is tiles_per_cta such warps that never synchronise with
// each other after the prologue.  The point of the shape is its shared-memory plan: the observation tile (the largest
// buffer, written only at the end) ALIASES the grid and inventory rows (read only until the lidar is done),
//     tile = header 128 B | region max(grid + inventory rows, observation tile)
// which is 8 KB on C2 instead of 13 KB.  All tiles of a one-wave launch then fit in HALF an SM (C2: 14 warps, 112 KB, one
// CTA per SM), so the NEXT launch of the stream — started early through programmatic dependent launch — is co-resident:
// its prologue, its zero-fill and (other handle: early_state) its TMA loads run underneath this launch's compute and
// store phases instead of after them.  Per warp:
//   load    two TMA bulk copies (grid rows, inventory rows) on the tile's mbarrier
//   step    all 32 lanes, no hand-over
//   store 1 inventory tile -> HBM (TMA bulk store, issued right after the step)
//   lidar   line gather into a RegSink: hits and inventory tail stay in registers
//   store 2 once the inventory store has read its rows: zero the region, write the <= 8 hits + tail per row, TMA bulk store
//   outputs pose / reward / step_cost / done / result straight from registers (lane = env: full lines), statistics
#define NGW_WTILE_HDR 128            // mbarrier (8) | dump word at +16
#define NGW_WCTA_HDR 384            // [0] tiles done | per-warp statistics partials at +64: int4[16]

// NT: compile-time bound of the inventory tail kept in registers (8 when every config has n_inv_obs <= 8, else 16)
template <int NC, int NT>
__global__ void __launch_bounds__(512, 2) step1w_kernel(const __grid_constant__ StepArgs<NC> args) {
    extern __shared__ __align__(128) unsigned char smem[];
    const StepParams& p = args.p;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int tile = (int)blockIdx.x * p.tiles_per_cta + wid;
    const bool active = tile < p.n_tiles;
    const long long e0 = p.env_begin + (long long)tile * 32;
    const long long e = e0 + lane;
    const bool valid = active && e < p.env_end;
    const bool full_tile = e0 + 32 <= p.env_end;
    const bool stepping = p.actions != nullptr;

    int* scta = reinterpret_cast<int*>(smem);
    uint8_t* sfirstk = smem + p.off_luts;
    int8_t* sslot = reinterpret_cast<int8_t*>(smem + p.off_luts + NGW_MAX_MAP_SIZE);
    unsigned char* gbase = smem + p.off_groups + wid * p.group_bytes;
    uint64_t* bar = reinterpret_cast<uint64_t*>(gbase);               // "tile landed" barrier
    unsigned char* region = gbase + NGW_WTILE_HDR;
    int8_t* smap = reinterpret_cast<int8_t*>(region);
    int32_t* sinv = reinterpret_cast<int32_t*>(region + p.map_bytes);
    unsigned char* sobs = region;                                     // aliases the rows above
    const uint32_t region_a = smem_u32(region);
    const uint32_t in_bytes = (uint32_t)(p.map_bytes + p.inv_bytes);
    const uint32_t obs_tile = p.obs != nullptr ? 32u * (uint32_t)p.obs_srow : 0u;

    // ---- prologue without global state
    if (threadIdx.x == 0) scta[0] = 0;
    if (lane == 0 && wid < p.tiles_per_cta) mbar_init(bar, 1);   // (the CTA's last warp is the gate warp: it owns no tile)
    stage_lidar_luts<NC>(args, sfirstk, sslot);
    __syncthreads();                                                  // the only CTA-wide barrier

    // The GATE warp (the CTA's last) keeps the stream's order: it waits for the preceding grid and only then lets the
    // next launch start, so at most two consecutive launches are ever in flight and this grid cannot complete before its
    // predecessor has.  In concurrent mode the tile warps below never wait: the two launches step different batches.
    if (wid == p.tiles_per_cta) {
        asm volatile("griddepcontrol.wait;" ::: "memory");
        asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
        return;
    }

    const int8_t* gmap = p.map + e0 * p.cells;
    int32_t* ginv = p.inv + e0 * p.inv_stride;
    const uint64_t pol_first = policy_evict_first();
    auto issue_loads = [&]() {
        if (lane == 0) issue_tile_loads(p, bar, smap, gmap, sinv, ginv, pol_first);
    };
    uchar4 ps = make_uchar4(0, 0, 0, 0);
    const bool early = p.early_state && active;
    if (early) {                                                      // see step1_kernel: this handle's state is complete already
        issue_loads();
        ps = __ldcg(&p.pose[e]);   // L2 only: launches overlap, an SM's L1 is not a safe place for another grid's data
    }
    // the part of the observation tile that lies beyond the rows it aliases is zeroed while the loads fly
    zero_span(region_a + in_bytes + (uint32_t)lane * 16u, region_a + obs_tile, 512u);
    if (!p.concurrent) asm volatile("griddepcontrol.wait;" ::: "memory");   // previous kernel of the stream done + visible
    // (the gate warp has let the dependent launch start by now or will: it is co-resident — half an SM per launch)
    if (!active) return;
    if (!early) {
        issue_loads();
        ps = __ldcg(&p.pose[e]);   // L2 only: launches overlap, an SM's L1 is not a safe place for another grid's data
    }

    const int cfg_i = (NC == 1) ? 0 : (int)__ldcg(&p.cfg_id[e]);
    const DevConfig& dc = args.config(cfg_i);
    const ngw_config& cfg = dc.c;
    int action = 0;
    if (stepping && valid) action = __ldcg(&p.actions[e]);

    mbar_wait(bar, 0);

    EnvRow env;
    env.m = smap + lane * p.cells;
    env.gm = p.map + e * p.cells;
    env.inv = sinv + lane * p.inv_stride;
    env.ms = p.ms;
    env.set_pose(ps);

    // ---- step
    uint32_t counts = 0;                                              // steps | episodes << 6 | successes << 12 | resets << 18 | invalid << 24
    StepOut o;
    o.clear();
    if (stepping) {
        int did_reset = 0;
        if (valid) {
            const ngw_action_entry a = decode_action(cfg, action);
            counts = 1u;
            if (a.op == NGW_OP_INVALID) {                             // wrappers.py:76 / pogostick_v1_env.py:236 would raise
                counts |= 1u << 24;
                atomicOr(&p.err[e], NGW_ERR_INVALID_ACTION);
            } else {
                step_env(env, cfg, a, o);
                did_reset = end_of_step(p, e, o);
                counts |= ((uint32_t)o.done << 6) | ((uint32_t)o.goal << 12) | ((uint32_t)did_reset << 18);
            }
            ps = env.pose();
        }
        if (p.auto_reset) queue_resets(p, lane, e, did_reset);       // queue the finished envs for reset_list_kernel
        // ---- store 1: the inventory tile leaves as soon as the step is done
        if (full_tile) {
            fence_async_smem();
            __syncwarp();
            if (lane == 0) { bulk_s2g(ginv, sinv, (uint32_t)p.inv_bytes); bulk_commit(); }
        } else {
            __syncwarp();
            copy16(ginv, sinv, p.inv_bytes, lane, 32);
        }
    }

    // ---- LidarInFront of the new state, into registers
    if (p.obs != nullptr) {
        RegSink<NT> sink;
        sink.init(p.obs_format);
        const bool look = valid && cfg.n_beams > 0;
        if (look) {
            const LidarLuts luts = lane_luts<NC>(p, sfirstk, sslot, cfg_i);
            lidar_lines<false, RegSink<NT> >(env, cfg, (NC > 0) ? args.cfg[0].lidar : dc.lidar, luts, sink, 0xF);
            obs_tail<RegSink<NT>, NT>(env, cfg, sink, dc.lidar.tail_first);
        }
        // ---- store 2: the rows have been consumed (and read by the inventory store) -> the region becomes the observation tile
        if (lane == 0) bulk_wait_read<0>();
        __syncwarp();
        zero_span(region_a + (uint32_t)lane * 16u, region_a + (in_bytes < obs_tile ? in_bytes : obs_tile), 512u);
        __syncwarp();
        if (look) {
            sink.flush(region_a + (uint32_t)(lane * p.obs_srow), smem_u32(gbase + 16), cfg.n_lidar_items,
                       obs_tail_offset(p.obs_format, cfg.n_lidar_items, cfg.n_beams), cfg.n_inv_obs);
        }
        if (full_tile) {
            fence_async_smem();
            __syncwarp();
            store_obs_tile(p, e0, sobs, lane, pol_first);
            bulk_commit();
        } else {
            __syncwarp();
            copy_obs_rows(p, e0, sobs, p.obs_srow, lane, 32);
        }
    }

    // ---- per-env outputs (lane = env: full lines) and episode statistics
    if (stepping) {
        if (valid) {
            p.pose[e] = ps;
            p.reward[e] = (float)o.reward;
            p.done[e] = (uint8_t)o.done;
            p.cost[e] = o.cost;
            p.result[e] = (uint8_t)o.result;
            if (p.msg != nullptr) p.msg[e] = (uint16_t)o.msg;
        }
        // warp reductions -> this warp's slot in shared memory; the last warp of the CTA to arrive folds the slots and
        // issues one set of global atomics per CTA
        const uint32_t c_all = __reduce_add_sync(0xFFFFFFFFu, counts);            // five counts <= 32: 6 bits apiece
        const int r_sum = __reduce_add_sync(0xFFFFFFFFu, o.reward);
        const float c_sum = warp_sum(o.cost);
        int4* slots = reinterpret_cast<int4*>(smem + 64);
        const int n_tiles_cta = min(p.tiles_per_cta, p.n_tiles - (int)blockIdx.x * p.tiles_per_cta);
        int last = 0;
        if (lane == 0) {
            slots[wid] = make_int4((int)c_all, r_sum, __float_as_int(c_sum), 0);
            __threadfence_block();
            last = atomicAdd(&scta[0], 1) == n_tiles_cta - 1;
        }
        if (__shfl_sync(0xFFFFFFFFu, last, 0)) {
            __threadfence_block();
            int4 v = make_int4(0, 0, 0, 0);
            if (lane < n_tiles_cta) {
                const volatile int* sv = reinterpret_cast<const volatile int*>(&slots[lane]);
                v.x = sv[0]; v.y = sv[1]; v.z = sv[2];
            }
            // counts of up to 16 warps x 32 lanes need 10 bits: widen before the second reduction
            const uint32_t lo = ((uint32_t)v.x & 63u) | ((((uint32_t)v.x >> 6) & 63u) << 10) | ((((uint32_t)v.x >> 12) & 63u) << 20);
            const uint32_t hi = (((uint32_t)v.x >> 18) & 63u) | ((((uint32_t)v.x >> 24) & 63u) << 10);
            const uint32_t a_tot = __reduce_add_sync(0xFFFFFFFFu, lo), b_tot = __reduce_add_sync(0xFFFFFFFFu, hi);
            const int r_tot = __reduce_add_sync(0xFFFFFFFFu, v.y);
            const float c_tot = warp_sum(__int_as_float(v.z));
            if (lane == 0) {
                const int n_step = a_tot & 1023, n_done = (a_tot >> 10) & 1023, n_succ = (a_tot >> 20) & 1023;
                const int n_reset = b_tot & 1023, n_inv = (b_tot >> 10) & 1023;
                flush_stats(p.stats, blockIdx.x, n_step - n_inv, r_tot, c_tot, n_done, n_succ, n_reset, n_inv);
            }
        }
    }
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    bulk_wait_read<0>();                                              // shared memory must outlive the bulk stores' reads
}

// ------------------------------------------------------------------ the K-STEP ROLLOUT kernel, LANE-PAIR shape
// (ngw_rollout / ngw_rollout_policy on grids up to 32x32 with the canonical 8-beam geometry; everything else takes
// rollout_kernel above.)  A rollout never leaves the SM between steps, so it is bound by the latency of one warp's
// dependent instruction chain, not by memory: 14 tiles per SM at one warp per tile issue ~0.35 instructions per cycle and
// scheduler.  Here a tile of 32 envs is stepped by TWO warps of 16 envs each, and every env is owned by a PAIR of lanes
// (l, l + 16): the low lane runs the step; for the LidarInFront observation each lane gathers two of the four lines
// through the agent — low lane row + column, high lane the two diagonals — in the SAME instruction stream (per-lane line
// base, stride and beam directions: no divergence); each lane accumulates the policy scores of its own <= 4 hits (and of
// every other inventory-tail entry), W rows read as 128-bit words, and one butterfly exchange adds the halves.
// Per-step statistics stay in registers and are folded once per launch.  The final observation tile aliases the
// grid / inventory rows like step1w_kernel's.
struct PairLine {
    const int8_t* p0;       // cell of the line in grid row 0 (row line: grid column 0)
    int stride;             // linear offset between consecutive cells of the line
    int pos;                // the agent's bit on the line
    uint32_t mask;          // bits whose cell lies inside the grid
    int a_pos, a_neg;       // compass directions of the two beams
};

template <int MS>
__device__ __forceinline__ uint32_t pair_gather(const PairLine& ln, int ms_rt) {
    const int ms = MS > 0 ? MS : ms_rt;
    const uint8_t* q = reinterpret_cast<const uint8_t*>(ln.p0);
    uint32_t occ = 0;
    if (MS > 0) {
#pragma unroll
        for (int i = 0; i < ms; i++) occ |= (q[i * ln.stride] != 0 ? 1u : 0u) << i;
    } else {
#pragma unroll 4
        for (int i = 0; i < ms; i++) occ |= (q[i * ln.stride] != 0 ? 1u : 0u) << i;
    }
    return occ & ln.mask;
}

// the two beams of one line -> (observation index << 8) | range (the policy's dot product), or with kSplit
// (beam << 16) | (lidar slot << 8) | range (observation rows of any layout); 0 = nothing reported
template <bool kSplit>
__device__ __forceinline__ void pair_beams(uint32_t occ, const PairLine& ln, const int8_t* here, bool diagonal, int K, int L,
                                           int rot, const LidarLuts& luts, uint32_t& hit_pos, uint32_t& hit_neg) {
    const int p = ln.pos;
    const uint32_t hi = (occ >> p) >> 1;
    const uint32_t lo = occ & ((1u << p) - 1u);
    const int n_pos = __ffs((int)hi);
    const int n_neg = lo != 0 ? p - (31 - __clz((int)lo)) : 0;
#pragma unroll
    for (int side = 0; side < 2; side++) {
        const int n = side ? n_neg : n_pos;
        const int a = side ? ln.a_neg : ln.a_pos;
        const int kd = (int)luts.firstk[n > 0 ? n - 1 : 0];
        const int k = diagonal ? kd : (n <= K ? n : 0);
        const int id = here[side ? -n * ln.stride : n * ln.stride];
        const int slot = luts.slot[id];                               // -1: occludes but is not a lidar item (Q2)
        const uint32_t at = kSplit ? ((uint32_t)((a - rot) & 7) << 8) | (uint32_t)slot : (uint32_t)(((a - rot) & 7) * L + slot);
        const uint32_t h = (slot >= 0 && n != 0 && k != 0) ? (at << 8) | (uint32_t)k : 0u;
        if (side) hit_neg = h; else hit_pos = h;
    }
}

// the four hits of this lane's two lines (half 0: row, column; half 1: diagonal, anti-diagonal), packed as pair_beams<kSplit>
template <int MS, bool kSplit>
__device__ __forceinline__ void pair_lidar(const EnvRow& e, const ngw_config& cfg, const LidarDev& t, const LidarLuts& luts,
                                           int half, uint32_t hit[4]) {
    const int ms = MS > 0 ? MS : e.ms;
    const int r = e.r, c = e.c;
    const uint32_t full = 0xFFFFFFFFu >> (32 - ms);
    const int dlo = r - c, alo = c + r - (ms - 1);
    PairLine l1, l2;
    l1.p0 = e.m + (half ? (c - r) : r * ms);      l1.stride = half ? ms + 1 : 1;   l1.pos = half ? r : c;
    l1.mask = half ? (dlo >= 0 ? (full << dlo) : (full >> (-dlo))) & full : full;
    l1.a_pos = half ? 1 : 2;                      l1.a_neg = half ? 5 : 6;
    l2.p0 = e.m + (half ? (c + r) : c);           l2.stride = half ? ms - 1 : ms;  l2.pos = r;
    l2.mask = half ? (alo >= 0 ? (full << alo) : (full >> (-alo))) & full : full;
    l2.a_pos = half ? 7 : 0;                      l2.a_neg = half ? 3 : 4;
    const uint32_t o1 = pair_gather<MS>(l1, ms), o2 = pair_gather<MS>(l2, ms);
    const int K = cfg.max_range, L = cfg.n_lidar_items;
    const int rot = (int)((*reinterpret_cast<const uint32_t*>(t.rot) >> (8 * e.facing)) & 7u);
    const int8_t* here = e.m + r * ms + c;
    pair_beams<kSplit>(o1, l1, here, half != 0, K, L, rot, luts, hit[0], hit[1]);
    pair_beams<kSplit>(o2, l2, here, half != 0, K, L, rot, luts, hit[2], hit[3]);
}

// score[a] += v * W[idx][a], a < 4 * A4; W rows are 16 * A4 bytes in shared memory
template <int A4>
__device__ __forceinline__ void policy_mac(int (&acc)[16], const int32_t* w, int idx, int v) {
    const int4* row = reinterpret_cast<const int4*>(w + idx * (4 * A4));
#pragma unroll
    for (int q = 0; q < A4; q++) {
        const int4 x = row[q];
        acc[4 * q] += v * x.x; acc[4 * q + 1] += v * x.y; acc[4 * q + 2] += v * x.z; acc[4 * q + 3] += v * x.w;
    }
}

#define NGW_R2_HDR 128
// A4: ceil(policy actions / 4) for the closed loop, 0 = actions given or drawn (no per-step observation)
template <int NC, int A4>
__global__ void __launch_bounds__(64, 14) rollout2_kernel(const __grid_constant__ StepArgs<NC> args) {
    extern __shared__ __align__(128) unsigned char smem[];
    const StepParams& p = args.p;
    const int lane = threadIdx.x & 31, g = threadIdx.x >> 5;
    const int half = lane >> 4, el = (lane & 15) + 16 * g;            // lane pair (l, l + 16) owns env el of the tile
    const bool low = half == 0;
    const long long e0 = p.env_begin + (long long)blockIdx.x * 32;
    const long long e = e0 + el;
    const bool valid = e < p.env_end;
    const bool full_tile = e0 + 32 <= p.env_end;

    uint64_t* bar = reinterpret_cast<uint64_t*>(smem);
    uint8_t* sfirstk = smem + p.off_luts;
    int8_t* sslot = reinterpret_cast<int8_t*>(smem + p.off_luts + NGW_MAX_MAP_SIZE);
    uint32_t* sscratch = reinterpret_cast<uint32_t*>(smem + p.off_scratch) + g * NGW_RESET_SCRATCH_WORDS;   // auto-reset, per warp
    int32_t* spol = reinterpret_cast<int32_t*>(smem + p.off_policy);  // bias [16] | W [obs_dim][4 * A4]
    unsigned char* region = smem + p.off_in;
    int8_t* smap = reinterpret_cast<int8_t*>(region);
    int32_t* sinv = reinterpret_cast<int32_t*>(region + p.map_bytes);
    unsigned char* sobs = region;                                     // aliases the rows above (written after the last step)
    const uint32_t in_bytes = (uint32_t)(p.map_bytes + p.inv_bytes);

    const int8_t* gmap = p.map + e0 * p.cells;
    int32_t* ginv = p.inv + e0 * p.inv_stride;
    if (threadIdx.x == 0) mbar_init(bar, 1);
    stage_lidar_luts<NC>(args, sfirstk, sslot);
    __syncthreads();
    asm volatile("griddepcontrol.wait;" ::: "memory");
    if (threadIdx.x == 0) {
        mbar_expect_tx(bar, in_bytes);
        bulk_g2s(smap, gmap, (uint32_t)p.map_bytes, bar);
        bulk_g2s(sinv, ginv, (uint32_t)p.inv_bytes, bar);
    }
    if (A4 > 0) {                                                     // policy: bias, then W with rows padded to 4 * A4 entries
        const int A = p.policy_actions, AP = A4 > 0 ? 4 * A4 : 4;
        for (int i = threadIdx.x; i < 16; i += 64) spol[i] = i < A ? p.policy_b[i] : 0;
        for (int i = threadIdx.x; i < p.obs_dim * AP; i += 64) {
            const int j = i / AP, a = i - j * AP;
            spol[16 + i] = a < A ? p.policy_w[j * A + a] : 0;
        }
    }
    const int cfg_i = (NC == 1) ? 0 : (int)p.cfg_id[valid ? e : e0];
    const DevConfig& dc = args.config(cfg_i);
    const ngw_config& cfg = dc.c;
    const LidarDev& geom = (NC > 0) ? args.cfg[0].lidar : dc.lidar;
    const LidarLuts luts = lane_luts<NC>(p, sfirstk, sslot, cfg_i);
    const bool given_actions = A4 == 0 && !p.random_policy;
    uchar4 ps = p.pose[valid ? e : e0];
    int action = 0;
    if (given_actions && valid && low) action = p.actions[e];
    mbar_wait(bar, 0);
    __syncthreads();                                                  // policy weights staged

    EnvRow env;
    env.m = smap + el * p.cells;
    env.gm = p.map + e * p.cells;
    env.inv = sinv + el * p.inv_stride;
    env.ms = p.ms;
    env.set_pose(ps);

    StepOut o;
    o.clear();
    float cost_sum = 0.0f;
    int reward_sum = 0, n_done = 0, n_succ = 0, n_reset = 0, n_invalid = 0;
    const int n_lidar = cfg.n_lidar_items * cfg.n_beams;
    RandomPolicy rpol;
    rpol.first = 0u; rpol.w[0] = rpol.w[1] = rpol.w[2] = rpol.w[3] = 0u;
    for (int t = 0; t < p.n_steps; t++) {
        int next_action = 0;
        if (given_actions && t + 1 < p.n_steps && valid && low) next_action = p.actions[(t + 1) * p.act_stride + e];
        if (A4 > 0) {                                                 // observe (two lines per lane), score, exchange, argmax
            int acc[16];
#pragma unroll
            for (int a = 0; a < 16; a++) acc[a] = (a < 4 * A4 && low) ? spol[a] : 0;
            if (cfg.n_beams > 0) {
                uint32_t hit[4];
                if (p.ms == 10) pair_lidar<10, false>(env, cfg, geom, luts, half, hit);
                else pair_lidar<0, false>(env, cfg, geom, luts, half, hit);
#pragma unroll
                for (int j = 0; j < 4; j++)
                    if (hit[j]) policy_mac<A4>(acc, spol + 16, (int)(hit[j] >> 8), (int)(hit[j] & 0xFFu));
                // inventory tail: entry i = 2 q + half
                const int n_tail = cfg.n_inv_obs, tf = dc.lidar.tail_first;
                for (int i = half; i < n_tail; i += 2) {
                    const int v = env.inv[tf >= 0 ? tf + i : (int)cfg.inv_obs_item[i]];
                    if (v != 0) policy_mac<A4>(acc, spol + 16, n_lidar + i, v);
                }
            }
#pragma unroll
            for (int a = 0; a < 4 * A4; a++) acc[a] += __shfl_xor_sync(0xFFFFFFFFu, acc[a], 16);
            const int n_valid = cfg.n_actions < p.policy_actions ? cfg.n_actions : p.policy_actions;
            int best = 0, best_v = acc[0];
#pragma unroll
            for (int a = 1; a < 4 * A4; a++) if (a < n_valid && acc[a] > best_v) { best_v = acc[a]; best = a; }
            action = best;
        } else if (p.random_policy && valid && low) {
            action = rpol.draw(p.policy_seed, (uint64_t)(p.first_gid + e), (uint32_t)t, (uint32_t)(cfg.n_actions > 0 ? cfg.n_actions : 1));
        }
        int did_reset = 0;
        __syncwarp();                                                 // the high lanes have read the rows
        if (valid && low) {
            if (p.actions_out != nullptr) p.actions_out[t * p.act_stride + e] = action;
            o.clear();
            // (decode_action, inlined by hand: the call shifts this kernel's spills)
            ngw_action_entry a;
            a.op = NGW_OP_INVALID;
            if (action >= 0 && action < cfg.n_actions) {
                uint2 raw = *reinterpret_cast<const uint2*>(&cfg.actions[action]);
                memcpy(&a, &raw, sizeof(a));
            }
            if (a.op == NGW_OP_INVALID) {
                n_invalid++;
                p.err[e] |= NGW_ERR_INVALID_ACTION;
            } else {
                step_env(env, cfg, a, o);
                n_succ += o.goal;
                int finished = o.done;
                if (p.max_episode_steps > 0) {
                    int len = p.ep_len[e] + 1;
                    if (len >= p.max_episode_steps) { finished = 1; o.done = 1; }
                    p.ep_len[e] = finished && p.auto_reset ? 0 : len;
                }
                if (finished && p.auto_reset) { did_reset = 1; n_reset++; }
            }
            reward_sum += o.reward; cost_sum += o.cost; n_done += o.done;
        }
        if (p.auto_reset) {
            if (__ballot_sync(0xFFFFFFFFu, did_reset) != 0) {         // regenerate in place, warp-cooperatively (this warp's 16 envs)
                uchar4 q = env.pose();
                auto_reset_warp(p, p.dcfgs, cfg_i, did_reset != 0, smap + 16 * g * p.cells, sinv + 16 * g * p.inv_stride,
                                sscratch, e0 + 16 * g, q);
                env.set_pose(q);
            }
        }
        // the pair's high lane follows the low lane's pose; the step's writes to the tile become visible to it
        {
            uint32_t pose = (uint32_t)env.r | ((uint32_t)env.c << 8) | ((uint32_t)env.facing << 16) | ((uint32_t)env.sel << 24);
            __syncwarp();
            pose = __shfl_sync(0xFFFFFFFFu, pose, lane & 15);
            env.r = pose & 0xFF; env.c = (pose >> 8) & 0xFF; env.facing = (pose >> 16) & 0xFF; env.sel = pose >> 24;
        }
        action = next_action;
    }

    // ---- outputs and statistics (low lanes own them)
    if (valid && low) {
        p.pose[e] = env.pose();
        p.reward[e] = (float)reward_sum;
        p.done[e] = (uint8_t)o.done;
        p.cost[e] = cost_sum;
        p.result[e] = (uint8_t)o.result;
        if (p.done_count != nullptr) p.done_count[e] = n_done;
        if (p.msg != nullptr) p.msg[e] = (uint16_t)o.msg;
    }
    const int steps = (valid && low) ? p.n_steps - n_invalid : 0;
    const int s_steps = __reduce_add_sync(0xFFFFFFFFu, steps), s_rew = __reduce_add_sync(0xFFFFFFFFu, reward_sum);
    const int s_done = __reduce_add_sync(0xFFFFFFFFu, n_done), s_succ = __reduce_add_sync(0xFFFFFFFFu, n_succ);
    const int s_reset = __reduce_add_sync(0xFFFFFFFFu, n_reset), s_inv = __reduce_add_sync(0xFFFFFFFFu, n_invalid);
    const float s_cost = warp_sum(cost_sum);
    if (lane == 0) flush_stats(p.stats, blockIdx.x, s_steps, s_rew, s_cost, s_done, s_succ, s_reset, s_inv);

    // ---- inventory tile out, final observation into the aliased region, observation tile out
    fence_async_smem();
    __syncthreads();                                                  // both warps are done stepping
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (full_tile) {
        if (threadIdx.x == 0) { bulk_s2g(ginv, sinv, (uint32_t)p.inv_bytes); bulk_commit(); }
    } else {
        copy16(ginv, sinv, p.inv_bytes, threadIdx.x, 64);
    }
    if (p.obs != nullptr) {
        uint32_t hit[4] = {0u, 0u, 0u, 0u};
        int32_t tail[NGW_REGSINK_TAIL];
        const bool look = valid && cfg.n_beams > 0;
        const int n_tail = cfg.n_inv_obs, tf = dc.lidar.tail_first;
        if (look) {
            if (p.ms == 10) pair_lidar<10, true>(env, cfg, geom, luts, half, hit);
            else pair_lidar<0, true>(env, cfg, geom, luts, half, hit);
#pragma unroll
            for (int i = 0; i < NGW_REGSINK_TAIL; i++)
                tail[i] = i < n_tail ? env.inv[tf >= 0 ? tf + i : (int)cfg.inv_obs_item[i]] : 0;
        }
        if (threadIdx.x == 0) bulk_wait_read<0>();
        __syncthreads();                                              // rows consumed by everyone (and by the inventory store)
        const uint32_t region_a = smem_u32(region);
        zero_span(region_a + threadIdx.x * 16u, region_a + (uint32_t)p.obs_bytes, 1024u);
        __syncthreads();
        if (look) {
            ObsRow orow;
            orow.p = sobs + el * p.obs_row_bytes;
            orow.fmt = p.obs_format;
#pragma unroll
            for (int j = 0; j < 4; j++)
                if (hit[j]) orow.put((int)(hit[j] >> 16), (int)((hit[j] >> 8) & 0xFFu), cfg.n_lidar_items, (int)(hit[j] & 0xFFu));
            if (low) {
                int32_t* tl = orow.tail(cfg.n_lidar_items, cfg.n_beams);
#pragma unroll
                for (int i = 0; i < NGW_REGSINK_TAIL; i++) if (i < n_tail) tl[i] = tail[i];
            }
        }
        if (full_tile) {
            fence_async_smem();
            __syncthreads();
            if (threadIdx.x == 0) {
                bulk_s2g_hint(p.obs + e0 * p.obs_row_bytes, sobs, (uint32_t)p.obs_bytes, policy_evict_first());
                bulk_commit();
            }
        } else {
            __syncthreads();
            // the rows are contiguous on both sides: one flat copy (copy_obs_rows costs this kernel spill stores)
            const int n = (int)((p.env_end - e0 < 32 ? p.env_end - e0 : 32)) * (p.obs_row_bytes >> 2);
            uint32_t* gobs = reinterpret_cast<uint32_t*>(p.obs + e0 * p.obs_row_bytes);
            const uint32_t* so = reinterpret_cast<const uint32_t*>(sobs);
            for (int i = threadIdx.x; i < n; i += 64) gobs[i] = so[i];
        }
    }
    if (threadIdx.x == 0) bulk_wait_read<0>();                        // shared memory must outlive the bulk stores' reads
}

}  // namespace ngw
