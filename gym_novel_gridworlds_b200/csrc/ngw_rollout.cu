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
    NGW_SMEM_ATTR((rollout_kernel<0>)); NGW_SMEM_ATTR((rollout_kernel<1>));
    NGW_SMEM_ATTR((rollout2_kernel<0, 0>)); NGW_SMEM_ATTR((rollout2_kernel<0, 1>)); NGW_SMEM_ATTR((rollout2_kernel<0, 2>));
    NGW_SMEM_ATTR((rollout2_kernel<0, 3>)); NGW_SMEM_ATTR((rollout2_kernel<0, 4>));
    NGW_SMEM_ATTR((rollout2_kernel<1, 0>)); NGW_SMEM_ATTR((rollout2_kernel<1, 1>)); NGW_SMEM_ATTR((rollout2_kernel<1, 2>));
    NGW_SMEM_ATTR((rollout2_kernel<1, 3>)); NGW_SMEM_ATTR((rollout2_kernel<1, 4>));
    return 0;
}

// K-step rollout launches (ngw_rollout / ngw_rollout_policy): one tile per CTA, tile resident across the steps
template <int NC>
static cudaError_t launch_rollout_nc(ngw_handle* h, StepParams p, cudaStream_t s) {
    // ---- shared-memory plan: header | lidar tables | reset scratch | grid + inventory tile | observation tile
    const int in_bytes = p.map_bytes + p.inv_bytes;
    p.off_luts = NGW_SMEM_HDR;
    p.off_scratch = p.off_luts + lut_bytes<NC>();
    p.off_policy = p.off_scratch + ((NGW_RESET_SCRATCH_WORDS * 4 + 127) & ~127);
    p.off_in = p.off_policy + (p.policy_w ? ((16 + p.obs_dim * p.policy_actions) * 4 + 127) & ~127 : 0);
    const long long tiles = (p.env_end - p.env_begin + 31) / 32;
    p.off_obs = p.off_in + in_bytes;
    const size_t smem = (size_t)p.off_obs + p.obs_bytes;
    // the K-step rollout is all step logic (one lidar pass at the end): one warp per tile keeps more tiles resident
    const int warps = (smem * 12 <= 227 * 1024) ? 1 : h->warps;
    claim_stream(h, s, false);
    return launch_tiles<NC>(rollout_kernel<NC>, h, p, dim3((unsigned)tiles), dim3(32 * warps), smem, s);
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
    const size_t smem = (size_t)p.off_in + (in_bytes > obs_tile ? in_bytes : obs_tile);
    if (smem > 200 * 1024) return cudaErrorNotSupported;
    const long long tiles = (p.env_end - p.env_begin + 31) / 32;
    claim_stream(h, s, false);
    return launch_tiles<NC>(rollout2_kernel<NC, A4>, h, p, dim3((unsigned)tiles), dim3(64), smem, s);
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
