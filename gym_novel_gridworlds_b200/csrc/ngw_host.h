// ngw_host.h — host-side declarations shared by the translation units of libngw_b200.so (ngw_capi.cu: handle, C-ABI, one-step
// launchers, cold kernels; ngw_rollout.cu: the K-step rollout launchers and their kernels — two units so that they compile
// in parallel).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include <string>
#include <vector>

#include "ngw_step.cuh"

using namespace ngw;

struct ngw_handle {
    int device = 0;
    long long n = 0, np = 0, first_gid = 0;
    unsigned long long seed = 0;
    int ms = 0, cells = 0, inv_stride = 0, obs_dim = 0, n_cfgs = 0;
    int map_bytes = 0, inv_bytes = 0, obs_bytes = 0, warps = 2, lidar_mode = 0;
    int obs_format = NGW_OBS_I32, obs_row_bytes = 0;   // observation row layout (ngw_set_obs_format)
    uint32_t key_mask = 0xFFFFFFFFu;
    bool lidar_uniform = false;
    bool concurrent = true;                        // independent consecutive launches may overlap (NGW_NO_CONCURRENT)
    DevConfig* d_cfgs = nullptr;
    std::vector<int16_t*> d_luts;
    std::vector<DevConfig> h_cfgs;
    int8_t* map = nullptr; uchar4* pose = nullptr; int32_t* inv = nullptr; uint8_t* cfg_id = nullptr;
    uint32_t* episode = nullptr; int32_t* ep_len = nullptr; uint32_t* err = nullptr; double* stats = nullptr;
    uint8_t* zero_byte = nullptr;
    uint16_t* msg = nullptr;                       // caller-owned message-code buffer (ngw_set_message_buffer)
    uint8_t* trunc = nullptr;                      // caller-owned episode-end buffers (ngw_set_episode_end_buffers): truncated
    unsigned char* final_obs = nullptr;            // flags, last observation rows of auto-reset envs
    ngw_rollout_record rec{};                      // caller-owned per-step record of the rollouts (ngw_set_rollout_record)
    bool rec_on = false;
    int32_t* reset_list = nullptr; int32_t* reset_ctl = nullptr;   // auto-reset queue; ctl[0] = count, ctl[1] = finished CTAs
    uint32_t* mt_key = nullptr; int32_t* mt_pos = nullptr;   // NGW_RNG_NUMPY: per-env np.random state (ngw_set_reset_rng)
    int sm_count = 148;
    long long launches = 0, concurrent_launches = 0;
    bool last_step_concurrent = false;             // the latest one-step launch overlapped its predecessor
    // host-buffer path: its own stream, ordered against the caller's streams with events
    cudaStream_t hs = nullptr;
    cudaEvent_t ev_dev = nullptr;                  // recorded on the caller's stream when the host path has to wait for it
    cudaStream_t last_dev_stream = nullptr;        // stream of the latest device-path call ...
    bool dev_dirty = false;                        // ... whose work the host stream has not been ordered after yet
    bool host_dirty = false;                       // host-path work enqueued and not yet waited for
    int32_t* h_actions = nullptr; unsigned char* h_obs = nullptr; size_t h_obs_bytes = 0; float* h_reward = nullptr;
    uint8_t* h_done = nullptr; float* h_cost = nullptr; uint8_t* h_result = nullptr;
};

struct MemRange { uintptr_t lo, hi; };
struct StreamTail {                       // the latest library launch on a stream
    ngw_handle* h = nullptr;
    unsigned long long cap_id = 0;        // stream capture it was recorded in, 0 = eager
    cudaGraphNode_t node = nullptr;       // its graph node (captures only)
    bool pure_step = false;               // 'gated': a one-step launch or the queued-reset kernel behind one — kernels that let
                                          // their dependents start only after everything before THEM has completed
    MemRange rd[2], wr[8];                // caller buffers it reads (actions) / writes (obs, reward, done, cost, result, msg,
                                          // truncated, final_obs)
    int n_rd = 0, n_wr = 0;
};

int fail(const std::string& m);
// see ngw_capi.cu
int claim_stream(ngw_handle* h, cudaStream_t s, bool want_early, const StreamTail* mine = nullptr, bool can_branch = false);
// ngw_rollout.cu
cudaError_t ngw_launch_rollout(ngw_handle* h, const StepParams& p, cudaStream_t s);
int ngw_rollout_set_attributes();
int ngw_rollout_record_fits(const ngw_handle* h, const StepParams& p);   // 0, or fail() with a message

// shared memory of the lidar tables a kernel with NC inline configs stages (stage_lidar_luts)
template <int NC>
constexpr int lut_bytes() { return (NGW_MAX_MAP_SIZE + NGW_MAX_ITEMS * (NC > 0 ? NC : 0) + 127) & ~127; }

template <int NC> void set_record(StepArgs<NC>&, const RecordParams*) {}
template <int NC> void set_record(RecArgs<NC>& a, const RecordParams* rec) { a.rec = *rec; }

// Launches a tile kernel with its argument block: the parameters plus the handle's first NC configs inline (and, for the
// recording rollout kernels, the record `rec`).
template <int NC, typename Args = StepArgs<NC> >
cudaError_t launch_tiles(void (*kernel)(Args), const ngw_handle* h, const StepParams& p, dim3 grid, dim3 block,
                         size_t smem, cudaStream_t s, const RecordParams* rec = nullptr) {
    static thread_local Args args;                  // host staging of the argument block (copied by the launch); per thread,
                                                    // so distinct handles stay independent across host threads
    args.p = p;
    for (int i = 0; i < NC && i < h->n_cfgs; i++) args.cfg[i] = h->h_cfgs[i];
    set_record(args, rec);
    cudaLaunchConfig_t lc;
    memset(&lc, 0, sizeof(lc));
    lc.gridDim = grid; lc.blockDim = block; lc.dynamicSmemBytes = smem;
    lc.stream = s;
    // PDL (trigger once a CTA's stores are issued, see the kernels): the next launch's prologue overlaps this launch's
    // store phase; C2 CUDA-graph replay 9.3 -> 8.6 us/step.  (An early trigger at kernel entry measured slower.)
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    lc.attrs = attr; lc.numAttrs = 1;
    return cudaLaunchKernelEx(&lc, kernel, args);
}
