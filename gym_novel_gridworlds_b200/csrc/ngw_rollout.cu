// ngw_rollout.cu — launchers of the K-step rollout kernels (ngw_rollout / ngw_rollout_policy): rollout2_kernel (lane pairs) and
// its fallback rollout_kernel.  A translation unit of its own: these are the largest kernels of the library.
#include "ngw_host.h"

#define NGW_SMEM_ATTR(K)                                                                                              \
    do {                                                                                                              \
        cudaError_t _e = cudaFuncSetAttribute(K, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);            \
        if (_e != cudaSuccess) return fail(std::string("cudaFuncSetAttribute(" #K "): ") + cudaGetErrorString(_e));   \
    } while (0)

// the rollout kernels' part of create_init's set_kernel_attributes (the kernels are instantiated in this unit)
int ngw_rollout_set_attributes() {
    // (rollout_kernel is the fallback behind rollout2_kernel: inline configs for one config, the global table otherwise)
    // (every kernel twice: without and with the per-step record, ngw_set_rollout_record)
    NGW_SMEM_ATTR((rollout_kernel<0, false>)); NGW_SMEM_ATTR((rollout_kernel<1, false>));
    NGW_SMEM_ATTR((rollout_kernel<0, true>)); NGW_SMEM_ATTR((rollout_kernel<1, true>));
    NGW_SMEM_ATTR((rollout2_kernel<0, 0, false>)); NGW_SMEM_ATTR((rollout2_kernel<0, 1, false>));
    NGW_SMEM_ATTR((rollout2_kernel<0, 2, false>)); NGW_SMEM_ATTR((rollout2_kernel<0, 3, false>));
    NGW_SMEM_ATTR((rollout2_kernel<0, 4, false>));
    NGW_SMEM_ATTR((rollout2_kernel<1, 0, false>)); NGW_SMEM_ATTR((rollout2_kernel<1, 1, false>));
    NGW_SMEM_ATTR((rollout2_kernel<1, 2, false>)); NGW_SMEM_ATTR((rollout2_kernel<1, 3, false>));
    NGW_SMEM_ATTR((rollout2_kernel<1, 4, false>));
    NGW_SMEM_ATTR((rollout2_kernel<0, 0, true>)); NGW_SMEM_ATTR((rollout2_kernel<0, 1, true>));
    NGW_SMEM_ATTR((rollout2_kernel<0, 2, true>)); NGW_SMEM_ATTR((rollout2_kernel<0, 3, true>));
    NGW_SMEM_ATTR((rollout2_kernel<0, 4, true>));
    NGW_SMEM_ATTR((rollout2_kernel<1, 0, true>)); NGW_SMEM_ATTR((rollout2_kernel<1, 1, true>));
    NGW_SMEM_ATTR((rollout2_kernel<1, 2, true>)); NGW_SMEM_ATTR((rollout2_kernel<1, 3, true>));
    NGW_SMEM_ATTR((rollout2_kernel<1, 4, true>));
    return 0;
}

// the handle's per-step record (p.record: ngw_set_rollout_record) as the recording kernels take it, its observation
// staging tile at shared-memory offset off_tile
static RecordParams record_params(const ngw_handle* h, int off_tile) {
    const ngw_rollout_record& r = h->rec;
    RecordParams rec;
    rec.obs = h->obs_dim > 0 ? static_cast<unsigned char*>(r.obs) : nullptr;
    rec.final_obs = h->obs_dim > 0 ? static_cast<unsigned char*>(r.final_obs) : nullptr;
    rec.reward = r.reward; rec.cost = r.step_cost; rec.done = r.done; rec.result = r.result; rec.trunc = r.truncated;
    rec.stride = h->np;
    rec.off_tile = off_tile;
    return rec;
}

// bytes of the record's observation staging tile (32 rows; none without a recorded observation)
static int record_tile_bytes(const RecordParams& rec, const StepParams& p) {
    return rec.obs != nullptr || rec.final_obs != nullptr ? 32 * p.obs_row_bytes : 0;
}

// numpy stream only: candidate lists for the `warps` warps that regenerate envs, appended at the plan's end `end`
static size_t numpy_lists(StepParams& p, size_t end, int warps) {
    if (p.mt_key == nullptr || !p.auto_reset) return end;
    p.off_lists = (int)((end + 127) & ~(size_t)127);
    return (size_t)p.off_lists + (size_t)warps * 2 * p.cells;
}

// rollout_kernel's shared-memory plan (offsets into p, the record's staging tile into rec) -> bytes per CTA
template <int NC>
static size_t rollout_plan(const ngw_handle* h, StepParams& p, RecordParams& rec) {
    // ---- header | lidar tables | reset scratch | grid + inventory tile | observation tile | record tile
    const int in_bytes = p.map_bytes + p.inv_bytes;
    p.off_luts = NGW_SMEM_HDR;
    p.off_scratch = p.off_luts + lut_bytes<NC>();
    p.off_policy = p.off_scratch + ((NGW_RESET_SCRATCH_WORDS * 4 + 127) & ~127);
    p.off_in = p.off_policy + (p.policy_w ? ((16 + p.obs_dim * p.policy_actions) * 4 + 127) & ~127 : 0);
    p.off_obs = p.off_in + in_bytes;
    rec = record_params(h, (p.off_obs + p.obs_bytes + 127) & ~127);
    const size_t end = p.record ? (size_t)rec.off_tile + record_tile_bytes(rec, p) : (size_t)p.off_obs + p.obs_bytes;
    return numpy_lists(p, end, 1);
}

// A rollout with a record runs rollout2_kernel where its plan fits 200 KB, else rollout_kernel, whose plan (grid,
// inventory and observation tiles plus the record's 32 staged rows) must fit a block's 227 KB of shared memory.
int ngw_rollout_record_fits(const ngw_handle* h, const StepParams& p) {
    StepParams q = p;
    RecordParams rec;
    const size_t smem = h->n_cfgs == 1 ? rollout_plan<1>(h, q, rec) : rollout_plan<0>(h, q, rec);
    if (smem <= 227 * 1024) return 0;
    return fail("rollout record: a tile with the record's " + std::to_string(record_tile_bytes(rec, p)) +
                " staged observation bytes needs " + std::to_string(smem) + " bytes of shared memory, more than a "
                "block's 227 KB (record fewer fields: no obs / final_obs, or narrower rows with ngw_set_obs_format)");
}

// K-step rollout launches (ngw_rollout / ngw_rollout_policy): one tile per CTA, tile resident across the steps
template <int NC>
static cudaError_t launch_rollout_nc(ngw_handle* h, StepParams p, cudaStream_t s) {
    RecordParams rec;
    const size_t smem = rollout_plan<NC>(h, p, rec);
    const long long tiles = (p.env_end - p.env_begin + 31) / 32;
    // the K-step rollout is all step logic (one lidar pass at the end): one warp per tile keeps more tiles resident
    const int warps = (smem * 12 <= 227 * 1024) ? 1 : h->warps;
    claim_stream(h, s, false);
    if (p.record)
        return launch_tiles<NC>(rollout_kernel<NC, true>, h, p, dim3((unsigned)tiles), dim3(32 * warps), smem, s, &rec);
    return launch_tiles<NC>(rollout_kernel<NC, false>, h, p, dim3((unsigned)tiles), dim3(32 * warps), smem, s);
}

// K-step rollout launches in the lane-pair shape (rollout2_kernel); cudaErrorNotSupported -> rollout_kernel
template <int NC, int A4>
static cudaError_t launch_rollout2_na(ngw_handle* h, StepParams p, cudaStream_t s) {
    const int in_bytes = p.map_bytes + p.inv_bytes;
    p.off_luts = NGW_R2_HDR;
    p.off_scratch = p.off_luts + lut_bytes<NC>();
    p.off_policy = p.off_scratch + (p.auto_reset ? ((2 * NGW_RESET_SCRATCH_WORDS * 4 + 127) & ~127) : 0);
    p.off_in = p.off_policy + (A4 > 0 ? ((16 + p.obs_dim * 4 * A4) * 4 + 127) & ~127 : 0);
    const int obs_tile = p.obs ? p.obs_bytes : 0;
    const RecordParams rec = record_params(h, (p.off_in + (in_bytes > obs_tile ? in_bytes : obs_tile) + 127) & ~127);
    const size_t smem = numpy_lists(p, p.record ? (size_t)rec.off_tile + record_tile_bytes(rec, p)
                                                : (size_t)p.off_in + (in_bytes > obs_tile ? in_bytes : obs_tile), 2);
    if (smem > 200 * 1024) return cudaErrorNotSupported;
    const long long tiles = (p.env_end - p.env_begin + 31) / 32;
    claim_stream(h, s, false);
    if (p.record) return launch_tiles<NC>(rollout2_kernel<NC, A4, true>, h, p, dim3((unsigned)tiles), dim3(64), smem, s, &rec);
    return launch_tiles<NC>(rollout2_kernel<NC, A4, false>, h, p, dim3((unsigned)tiles), dim3(64), smem, s);
}

template <int NC>
static cudaError_t launch_rollout2_nc(ngw_handle* h, const StepParams& p, cudaStream_t s) {
    if (h->ms > 32) return cudaErrorNotSupported;
    if (h->obs_dim > 0 && h->lidar_mode != 1) return cudaErrorNotSupported;
    for (const DevConfig& dc : h->h_cfgs)
        if (dc.c.n_inv_obs > NGW_REGSINK_TAIL) return cudaErrorNotSupported;
    if (p.policy_w == nullptr) return launch_rollout2_na<NC, 0>(h, p, s);
    switch ((p.policy_actions + 3) / 4) {
        case 1: return launch_rollout2_na<NC, 1>(h, p, s);
        case 2: return launch_rollout2_na<NC, 2>(h, p, s);
        case 3: return launch_rollout2_na<NC, 3>(h, p, s);
        default: return launch_rollout2_na<NC, 4>(h, p, s);
    }
}

cudaError_t ngw_launch_rollout(ngw_handle* h, const StepParams& p, cudaStream_t s) {
    const int nc = h->n_cfgs;
    cudaError_t e = nc == 1 ? launch_rollout2_nc<1>(h, p, s) : launch_rollout2_nc<0>(h, p, s);
    if (e != cudaErrorNotSupported) return e;
    if (nc == 1) return launch_rollout_nc<1>(h, p, s);
    return launch_rollout_nc<0>(h, p, s);
}
