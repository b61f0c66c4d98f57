// ngw_reset.cuh — the cold kernels of libngw_b200.so: Philox reset (one warp per env), the auto-reset queue consumer,
// masked observation, AgentMap crop, config-id conversion, statistics fold.
#pragma once
#include "ngw_step.cuh"

namespace ngw {

// ------------------------------------------------------------------ cold-path kernels (one thread per env, global memory)
struct ResetParams {
    const DevConfig* dcfgs;
    int8_t* map;
    uchar4* pose;
    int32_t* inv;
    const uint8_t* cfg_id;
    uint32_t* episode;
    int32_t* ep_len;
    uint32_t* err;
    const uint8_t* mask;
    long long n_envs, first_gid;
    unsigned long long seed;
    int ms, cells, inv_stride;
    int phase;   // 0: base + ops before the reset observation, 1: ops after it, 2: everything
    const uint8_t* zero_byte;   // a global byte that always reads 0 (see lidar_observe)
    const int32_t* reset_list;  // reset_list_kernel: queue written by the step kernel
    int32_t* reset_count;
    int32_t* done_ctas;
    unsigned char* obs;         // observation rows of obs_row_bytes bytes (layout as in the step kernel)
    unsigned char* final_obs;   // reset_list_kernel, optional: a regenerated env's row of obs is copied here before it is replaced
    int obs_dim, obs_row_bytes, obs_format;
    uint32_t key_mask;          // 0xFFFFFFFF; test knob NGW_DEBUG_KEY_MASK forces ties between the subset-sampling keys
    uint32_t* mt_key;           // NGW_RNG_NUMPY: the envs' np.random states, key [n][624] and pos [n]; nullptr = Philox
    int32_t* mt_pos;
};

#define NGW_RESET_WARPS 4
// The cold kernels regenerate an env on a shared-memory copy of its rows (every pass of reset_env_warp would otherwise
// pay HBM latency) and write the rows back with coalesced stores.
struct ResetScratch {
    uint32_t hist[NGW_RESET_SCRATCH_WORDS];
    int32_t inv[NGW_MAX_ITEMS];
    int8_t row[NGW_MAX_MAP_SIZE * NGW_MAX_MAP_SIZE];
};

__device__ __forceinline__ void rows_to_smem(ResetScratch& sc, const int8_t* m, const int32_t* inv, int cells, int inv_stride,
                                             int lane) {
    for (int i = lane; i < cells; i += 32) sc.row[i] = m[i];
    for (int i = lane; i < inv_stride; i += 32) sc.inv[i] = inv[i];
    __syncwarp();
}
__device__ __forceinline__ void rows_from_smem(const ResetScratch& sc, int8_t* m, int32_t* inv, int cells, int inv_stride,
                                               int lane) {
    __syncwarp();
    for (int i = lane; i < cells; i += 32) m[i] = sc.row[i];
    for (int i = lane; i < inv_stride; i += 32) inv[i] = sc.inv[i];
}

// With the numpy stream (p.mt_key) each warp also owns `cells` uint16 of dynamic shared memory for its candidate lists.
__global__ void __launch_bounds__(32 * NGW_RESET_WARPS) reset_kernel(const ResetParams p) {
    __shared__ ResetScratch scratch[NGW_RESET_WARPS];
    extern __shared__ __align__(16) uint16_t rk_lists[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    long long e = (long long)blockIdx.x * NGW_RESET_WARPS + warp;       // one warp regenerates one env
    if (e >= p.n_envs) return;
    if (p.mask != nullptr && p.mask[e] == 0) return;
    // numpy stream: a phase 0 that failed ended the reset program (the reference raised there)
    if (p.mt_key != nullptr && p.phase == 1 && (p.err[e] & NGW_ERR_PLACEMENT)) return;
    ResetScratch& sc = scratch[warp];
    const ngw_config* cfg = &p.dcfgs[p.cfg_id[e]].c;
    uchar4 ps = p.pose[e];
    int r = ps.x, c = ps.y, f = ps.z, sel = ps.w;
    uint64_t gid = (uint64_t)(p.first_gid + e);
    int k = cfg->reset_obs_after_ops;
    int8_t* m = p.map + e * p.cells;
    int32_t* inv = p.inv + e * p.inv_stride;
    uint32_t err;
    if (p.phase != 1) {
        uint32_t ep = p.episode[e] + 1;
        __syncwarp();
        const int end = p.phase == 0 ? k : NGW_MAX_RESET_OPS;
        if (p.mt_key != nullptr)
            err = reset_env_numpy_warp(cfg, sc.row, sc.inv, p.ms, p.inv_stride, p.mt_key + e * NGW_MT_WORDS, p.mt_pos + e,
                                       true, 0, end, rk_lists + warp * p.cells, r, c, f, sel);
        else
            err = reset_env_warp(cfg, sc.row, sc.inv, p.ms, p.inv_stride, p.seed, gid, ep, true, 0, end, sc.hist, r, c, f,
                                 sel, p.key_mask);
        if (lane == 0) { p.episode[e] = ep; p.ep_len[e] = 0; }
    } else {
        uint32_t ep = p.episode[e];
        rows_to_smem(sc, m, inv, p.cells, p.inv_stride, lane);
        if (p.mt_key != nullptr)
            err = reset_env_numpy_warp(cfg, sc.row, sc.inv, p.ms, p.inv_stride, p.mt_key + e * NGW_MT_WORDS, p.mt_pos + e,
                                       false, k, NGW_MAX_RESET_OPS, rk_lists + warp * p.cells, r, c, f, sel);
        else
            err = reset_env_warp(cfg, sc.row, sc.inv, p.ms, p.inv_stride, p.seed, gid, ep, false, k, NGW_MAX_RESET_OPS,
                                 sc.hist, r, c, f, sel, p.key_mask);
    }
    // a reset assigns the env's flags; its phase 1 adds those of the ops after the observation to what phase 0 assigned
    if (lane == 0) p.err[e] = p.phase == 1 ? p.err[e] | err : err;
    rows_from_smem(sc, m, inv, p.cells, p.inv_stride, lane);
    if (lane == 0) p.pose[e] = make_uchar4((unsigned char)r, (unsigned char)c, (unsigned char)f, (unsigned char)sel);
}

// NGW_RNG_NUMPY seeding: env e's state becomes np.random.seed(seed0 + e)'s (init_genrand, pos = 624)
__global__ void mt_seed_kernel(uint32_t* key, int32_t* pos, long long n, unsigned long long seed0) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    uint32_t s = (uint32_t)(seed0 + (unsigned long long)e);
    uint32_t* k = key + e * NGW_MT_WORDS;
    for (int i = 0; i < NGW_MT_WORDS; i++) {
        k[i] = s;
        s = 1812433253u * (s ^ (s >> 30)) + (uint32_t)i + 1u;
    }
    pos[e] = NGW_MT_WORDS;
}

// Second half of the single-step auto-reset: a grid-stride loop of warps over the queue the step kernel filled.  Each
// warp regenerates one env on a shared-memory copy of its rows (reset_env_warp), casts its LidarInFront beams into its
// observation row and writes the rows back.  Like ngw_reset, the observation of the new episode is taken after
// reset_obs_after_ops ops (quirk Q3: a novelty wrapped outside LidarInFront patches the state after the observation
// was computed).  The last CTA to finish empties the queue for the next step.
// (Measured and rejected: a whole CTA of 4 warps per env — at 96 registers only 5 such CTAs fit an SM, the
// ~2000 queued envs of a C5 step then take three rounds instead of one: 356 vs 315 us per step.)
// Shared memory is sized for the batch's grid (dynamic: NGW_RESET_WARPS x reset_list_scratch_bytes(cells)), so that one
// CTA of this kernel fits next to a full set of step CTAs when the next handle's step overlaps it (C5: 11 KB).
// With the numpy stream a warp's scratch also holds its candidate list: cells uint16 more.
__host__ __device__ inline int reset_list_scratch_bytes(int cells, bool numpy = false) {
    return NGW_RESET_SCRATCH_WORDS * 4 + NGW_MAX_ITEMS * 4 + ((cells + 15) & ~15) + (numpy ? (2 * cells + 15) & ~15 : 0);
}
struct ResetScratchView { uint32_t* hist; int32_t* inv; int8_t* row; };

__global__ void __launch_bounds__(32 * NGW_RESET_WARPS) reset_list_kernel(const ResetParams p) {
    extern __shared__ __align__(16) unsigned char rl_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    ResetScratchView sc;
    {
        unsigned char* base = rl_smem + warp * reset_list_scratch_bytes(p.cells, p.mt_key != nullptr);
        sc.hist = reinterpret_cast<uint32_t*>(base);
        sc.inv = reinterpret_cast<int32_t*>(base + NGW_RESET_SCRATCH_WORDS * 4);
        sc.row = reinterpret_cast<int8_t*>(base + NGW_RESET_SCRATCH_WORDS * 4 + NGW_MAX_ITEMS * 4);
    }
    // This kernel is launched plainly, so everything before it has completed; the stream's next launch (another handle's
    // step, if it can prove its independence) may start now and overlap the resets.
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    const int count = *reinterpret_cast<volatile int32_t*>(p.reset_count);
    for (int i = blockIdx.x * NGW_RESET_WARPS + warp; i < count; i += gridDim.x * NGW_RESET_WARPS) {
        const long long e = p.reset_list[i];
        const DevConfig& dc = p.dcfgs[p.cfg_id[e]];
        uchar4 ps = p.pose[e];
        int r = ps.x, c = ps.y, f = ps.z, sel = ps.w;
        int8_t* m = p.map + e * p.cells;
        int32_t* inv = p.inv + e * p.inv_stride;
        const uint64_t gid = (uint64_t)(p.first_gid + e);
        uint32_t ep = p.episode[e] + 1;
        __syncwarp();
        int k_obs = dc.c.reset_obs_after_ops;
        if (p.obs == nullptr || k_obs >= dc.c.n_reset_ops) k_obs = NGW_MAX_RESET_OPS;
        uint16_t* list = reinterpret_cast<uint16_t*>(sc.row + ((p.cells + 15) & ~15));   // numpy stream only
        uint32_t err = p.mt_key != nullptr
            ? reset_env_numpy_warp(&dc.c, sc.row, sc.inv, p.ms, p.inv_stride, p.mt_key + e * NGW_MT_WORDS, p.mt_pos + e,
                                   true, 0, k_obs, list, r, c, f, sel)
            : reset_env_warp(&dc.c, sc.row, sc.inv, p.ms, p.inv_stride, p.seed, gid, ep, true, 0, k_obs, sc.hist, r, c, f,
                             sel, p.key_mask);
        if (p.obs != nullptr) {                                       // observation of the new episode replaces the row
            ObsRow orow;
            orow.p = p.obs + e * p.obs_row_bytes;
            orow.fmt = p.obs_format;
            uint32_t* row = reinterpret_cast<uint32_t*>(orow.p);
            if (p.final_obs != nullptr) {                             // the finished episode's last observation is kept
                uint32_t* frow = reinterpret_cast<uint32_t*>(p.final_obs + e * p.obs_row_bytes);
                for (int k = lane; k < (p.obs_row_bytes >> 2); k += 32) frow[k] = row[k];
            }
            for (int k = lane; k < (p.obs_row_bytes >> 2); k += 32) row[k] = 0;
            if (lane == 0) sc.hist[0] = 0;                                // a shared-memory byte that reads 0
            __syncwarp();
            EnvRow env;                                                   // lidar on the shared-memory copy
            env.m = sc.row; env.gm = nullptr; env.inv = sc.inv; env.ms = p.ms;
            env.r = r; env.c = c; env.facing = f; env.sel = sel;
            const int8_t* zero = reinterpret_cast<const int8_t*>(sc.hist);
            LidarLuts luts;
            luts.slot = dc.c.lidar_slot; luts.firstk = dc.lidar.firstk;
            if (dc.c.n_beams > 0) {
                if (dc.lidar.lines) { if (lane < 4) lidar_observe<true>(env, dc, dc.lidar, luts, orow, zero, lane, 4, lane == 3); }
                else if (dc.lidar.fast) { if (lane < 8) lidar_observe<true>(env, dc, dc.lidar, luts, orow, zero, lane, 8, lane == 7); }
                else if (lane == 0) lidar_observe<true>(env, dc, dc.lidar, luts, orow, zero, 0, 1, true);
            }
            __syncwarp();
        }
        if (k_obs < dc.c.n_reset_ops && p.mt_key != nullptr && !(err & NGW_ERR_PLACEMENT))
            err |= reset_env_numpy_warp(&dc.c, sc.row, sc.inv, p.ms, p.inv_stride, p.mt_key + e * NGW_MT_WORDS,
                                        p.mt_pos + e, false, k_obs, NGW_MAX_RESET_OPS, list, r, c, f, sel);
        else if (k_obs < dc.c.n_reset_ops && p.mt_key == nullptr)
            err |= reset_env_warp(&dc.c, sc.row, sc.inv, p.ms, p.inv_stride, p.seed, gid, ep, false, k_obs,
                                  NGW_MAX_RESET_OPS, sc.hist, r, c, f, sel, p.key_mask);
        __syncwarp();
        for (int k = lane; k < p.cells; k += 32) m[k] = sc.row[k];
        for (int k = lane; k < p.inv_stride; k += 32) inv[k] = sc.inv[k];
        if (lane == 0) {
            p.episode[e] = ep;
            p.pose[e] = make_uchar4((unsigned char)r, (unsigned char)c, (unsigned char)f, (unsigned char)sel);
            if (err) p.err[e] |= err;
        }
        __syncwarp();
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(p.done_ctas, 1) == (int)gridDim.x - 1) { *p.reset_count = 0; *p.done_ctas = 0; }
    }
}

__global__ void observe_masked_kernel(const ResetParams p) {
    long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= p.n_envs) return;
    if (p.mask != nullptr && p.mask[e] == 0) return;
    const DevConfig& dc = p.dcfgs[p.cfg_id[e]];
    EnvRow env;
    env.m = p.map + e * p.cells;
    env.gm = nullptr;
    env.inv = p.inv + e * p.inv_stride;
    env.ms = p.ms;
    env.set_pose(p.pose[e]);
    ObsRow orow;
    orow.p = p.obs + e * p.obs_row_bytes;
    orow.fmt = p.obs_format;
    uint32_t* row = reinterpret_cast<uint32_t*>(orow.p);
    for (int i = 0; i < (p.obs_row_bytes >> 2); i++) row[i] = 0;
    LidarLuts luts;
    luts.slot = dc.c.lidar_slot; luts.firstk = dc.lidar.firstk;
    if (dc.c.n_beams > 0)
        lidar_observe<true>(env, dc, dc.lidar, luts, orow, reinterpret_cast<const int8_t*>(p.zero_byte), 0, 1, true);
}

// AgentMap.get_agentView (observation_wrappers.py:98-118): zero-padded (2v+1)^2 crop centred on the agent
__global__ void agent_map_kernel(const int8_t* map, const uchar4* pose, int8_t* out, long long n, int ms, int view) {
    const int side = 2 * view + 1;
    long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n * side * side) return;
    long long e = idx / (side * side);
    int k = (int)(idx - e * side * side);
    int r = pose[e].x - view + k / side, c = pose[e].y - view + k % side;
    out[idx] = (r >= 0 && r < ms && c >= 0 && c < ms) ? map[e * ms * ms + r * ms + c] : (int8_t)0;
}

__global__ void set_cfg_kernel(const int32_t* src, uint8_t* dst, long long n, int n_cfgs, uint32_t* err) {
    long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    int v = src ? src[e] : 0;
    if (v < 0 || v >= n_cfgs) { v = 0; err[e] |= 0x80000000u; }
    dst[e] = (uint8_t)v;
}

__global__ void stats_fold_kernel(double* slots, double* out, int reset_after) {
    int k = threadIdx.x;
    if (k >= NGW_STAT_COUNT) return;
    double s = 0.0;
    for (int i = 0; i < NGW_STAT_SLOTS; i++) {
        s += slots[i * NGW_STAT_COUNT + k];
        if (reset_after) slots[i * NGW_STAT_COUNT + k] = 0.0;
    }
    out[k] = s;
}

}  // namespace ngw
