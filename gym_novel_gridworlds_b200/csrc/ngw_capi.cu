// ngw_capi.cu — handle management and the extern "C" entry points of libngw_b200.so (include/ngw.h is the contract).
// The kernels live in ngw_step.cuh (hot path) and ngw_reset.cuh (cold paths); per-env device code in ngw_device.cuh.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "ngw_host.h"
#include "ngw_reset.cuh"


// ====================================================================== host side: handle + C-ABI
using namespace ngw;

static thread_local std::string g_err;
int fail(const std::string& m) { g_err = m; return 1; }
#define CK(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t _e = (call);                                                                         \
        if (_e != cudaSuccess) return fail(std::string(#call) + ": " + cudaGetErrorString(_e));          \
    } while (0)



// Device-path entry points run on the caller's stream, the host-buffer path on the handle's own non-blocking stream.
// These two keep them ordered: a device-path call first waits for unfinished host-path work, and the host path waits
// (on the device, through an event) for everything the latest device-path stream had been given.
// Which handle issued the latest state-WRITING launch on a stream (step / rollout / reset / load_state / set_env_configs).
// A one-step launch whose predecessor on its stream belongs to another handle may load its state before
// griddepcontrol.wait (see step1_kernel): its own last writer is at least two launches back, and the predecessor — one
// of this library's kernels, which trigger their dependents only after their own wait — cannot have started its body
// before that writer had completed.  Launches the library cannot see (the caller's own kernels, copies) only add
// distance.  The first launch of a stream capture is always conservative: a graph can be replayed after anything.
//
// Capture chains.  Inside a stream capture, a run of consecutive stepping one-step launches (nothing else captured
// between them: the stream's dependency set is exactly the one the library left after the previous launch) is spread
// over kBranches parallel branches of the graph.  The k-th handle to appear in the chain is pinned to branch
// k % kBranches; its launch depends only on the tip of that branch (the branch's first launch: on the chain's base, the
// dependency set the chain started from), and after every launch the stream's dependency set is restored to every
// branch's tip, so whatever the caller captures next (a kernel, an event record, the end of the capture) waits for all of
// them.  Branches are unordered against each other, so a launch joins a branch only if its caller buffers (launch_tail)
// do not conflict with those of any launch already on ANOTHER branch of the chain; otherwise, and for every other
// library launch, the chain ends there (the launch depends on every tip).  Within a branch the proof above holds with
// "the stream" read as "the branch": a handle's state is only ever written on its own branch, so the branch predecessor
// of another handle is gated behind that handle's last writer exactly as the stream predecessor is without branches.
// With as many branches as handles or more, every launch of a branch belongs to the same handle and waits (mode 0).
// Only one-wave launches branch (see branchable).
// W, measured on one B200 (1000 W power limit, 1965 MHz max SM clock) with bench.py's C2 line (18 rotating 65,536-env
// batches, 1008-launch graphs): 4.88 / 4.89 / 4.82 us per step with W = 2 / 3 / 4, against 5.97 without branches —
// no W beats another beyond the run-to-run spread; 3 is the shape of bench.py's `overlapped` arm (4.88 there).
static const int kBranches = 3;

struct Branch {
    StreamTail tail;                      // its latest launch; tail.node is the branch's tip
    std::vector<MemRange> rd, wr;         // caller buffers of every launch placed on it in this chain
};
struct Chain {
    bool active = false;
    std::vector<cudaGraphNode_t> base;    // the dependency set the chain started from,
    StreamTail base_tail;                 // the stream's latest launch at that point
    std::vector<ngw_handle*> base_block;  // and the handles whose launches may be nodes of the base
    std::vector<ngw_handle*> pinned;      // pinned[k] runs on branch k % kBranches
    Branch br[kBranches];
    int n_br = 0;                         // branches started
    int last = -1;                        // branch of the chain's latest launch
    std::vector<cudaGraphNode_t> left;    // the dependency set the library left after it: every branch's tip
};
struct StreamRec {
    StreamTail tail;                      // the latest library launch on the stream
    Chain chain;
};

static std::mutex g_order_mu;
static std::unordered_map<cudaStream_t, StreamRec> g_streams;
static thread_local bool g_first_in_capture = false; // the latest claim_stream saw the first library launch of a stream capture
static thread_local bool g_capturing = false;        // capture state of the stream seen by the latest claim_stream of this thread
static thread_local bool g_adjacent_hint = false;   // ngw_step_many: this launch directly follows the library's previous launch on the stream
static thread_local int g_branch = -1;               // branch of the chain the latest claim_stream placed its launch on, -1: none
static thread_local bool g_branch_head = false;      // ... the first launch of a branch other than the chain's first
static thread_local bool g_cross_branch = false;     // ... a branch other than its stream predecessor's

static bool overlaps(const MemRange* a, int na, const MemRange* b, int nb) {
    for (int i = 0; i < na; i++)
        for (int j = 0; j < nb; j++)
            if (a[i].lo < b[j].hi && b[j].lo < a[i].hi) return true;
    return false;
}

static bool same_set(const std::vector<cudaGraphNode_t>& a, const std::vector<cudaGraphNode_t>& b) {
    if (a.size() != b.size()) return false;
    for (cudaGraphNode_t x : a) {
        bool found = false;
        for (cudaGraphNode_t y : b) found |= x == y;
        if (!found) return false;
    }
    return true;
}

static bool contains(const std::vector<ngw_handle*>& v, const ngw_handle* h) {
    for (const ngw_handle* x : v) if (x == h) return true;
    return false;
}

static void add_ranges(std::vector<MemRange>& to, const MemRange* r, int n) {
    for (int i = 0; i < n; i++) {
        bool known = false;
        for (const MemRange& x : to) known |= x.lo <= r[i].lo && r[i].hi <= x.hi;
        if (!known) to.push_back(r[i]);
    }
}

// a read of one branch of what another writes, or two writes of one buffer
static bool conflicts(const StreamTail& mine, const Branch& other) {
    const int nr = (int)other.rd.size(), nw = (int)other.wr.size();
    return overlaps(mine.wr, mine.n_wr, other.wr.data(), nw) || overlaps(mine.wr, mine.n_wr, other.rd.data(), nr) ||
           overlaps(mine.rd, mine.n_rd, other.wr.data(), nw);
}

// Mode of a launch against its predecessor t: 0 (conservative), 1 (state loads may precede griddepcontrol.wait) or 2
// (independent of it: see step1w_kernel's gate warp).  `blocked`: a launch of this handle may be a direct predecessor.
// 2 needs PROOF that nothing sits between the two launches (`adjacent`: the dependency set is exactly t's graph node, or
// one call issued both), that t is a plain one-step launch of ANOTHER handle, and that the caller buffers of the two do
// not overlap.  Then everything this launch reads besides its own state (the actions) was complete before t was let go
// by ITS gate.
static int launch_mode(const StreamTail& t, bool blocked, unsigned long long cap_id, bool adjacent, const StreamTail* mine) {
    if (t.h == nullptr || blocked || t.cap_id != cap_id) return 0;
    if (mine != nullptr && t.pure_step && adjacent &&
        !overlaps(mine->wr, mine->n_wr, t.wr, t.n_wr) && !overlaps(mine->wr, mine->n_wr, t.rd, t.n_rd) &&
        !overlaps(mine->rd, mine->n_rd, t.wr, t.n_wr))
        return 2;
    return 1;
}

// Returns the launch's mode (launch_mode) and, for a stepping one-step launch inside a capture (`can_branch`), places it on
// a branch of the stream's capture chain: the stream's dependency set is then that branch's predecessor until
// join_branches.
int claim_stream(ngw_handle* h, cudaStream_t s, bool want_early, const StreamTail* mine, bool can_branch) {
    unsigned long long cap_id = 0;
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    const cudaGraphNode_t* d = nullptr;
    size_t n_d = 0;
    if (cudaStreamGetCaptureInfo(s, &cap, &cap_id, nullptr, &d, &n_d) != cudaSuccess) {
        cudaGetLastError(); cap = cudaStreamCaptureStatusNone; n_d = 0;
    }
    if (cap != cudaStreamCaptureStatusActive) { cap_id = 0; n_d = 0; }
    g_capturing = cap == cudaStreamCaptureStatusActive;
    const std::vector<cudaGraphNode_t> deps(d, d + n_d);
    g_branch = -1; g_branch_head = false; g_cross_branch = false;
    std::lock_guard<std::mutex> lk(g_order_mu);
    StreamRec& r = g_streams[s];
    const StreamTail t = r.tail;
    Chain& c = r.chain;
    g_first_in_capture = cap_id != 0 && t.cap_id != cap_id;
    // A chain of this capture that no library launch has ended yet: every handle it pinned may own a node of the current
    // dependency set — its tips — even when something else joined the set (a wait on another stream of the capture).
    const bool in_chain = c.active && cap_id != 0 && t.cap_id == cap_id;
    const bool chained = in_chain && same_set(deps, c.left);
    can_branch = can_branch && cap_id != 0 && mine != nullptr && h->concurrent;
    int mode = 0, b = -1, pin = -1;
    if (can_branch && chained) {
        for (int k = 0; k < (int)c.pinned.size() && pin < 0; k++) if (c.pinned[k] == h) pin = k;
        b = (pin >= 0 ? pin : (int)c.pinned.size()) % kBranches;
        for (int o = 0; o < c.n_br && b >= 0; o++)
            if (o != b && conflicts(*mine, c.br[o])) b = -1;
    }
    if (can_branch && b < 0) {            // a new chain starts at this launch, from the current dependency set
        Chain n;
        n.active = true; n.base = deps; n.base_tail = t;
        n.base_block = in_chain ? c.pinned : std::vector<ngw_handle*>{};
        n.base_block.push_back(t.h);
        c = n;
        b = 0; pin = -1;
    }
    if (b >= 0) {
        const bool head = b >= c.n_br;
        const StreamTail& pred = head ? c.base_tail : c.br[b].tail;
        std::vector<cudaGraphNode_t> pd = head ? c.base : std::vector<cudaGraphNode_t>{pred.node};
        if (!same_set(pd, deps) &&
            cudaStreamUpdateCaptureDependencies(s, pd.data(), pd.size(), cudaStreamSetCaptureDependencies) != cudaSuccess) {
            cudaGetLastError();
            c.active = false; b = -1;     // (the dependency set is unchanged: the launch joins every tip)
        } else {
            const bool blocked = head ? contains(c.base_block, h) : pred.h == h;
            const bool adjacent = pd.size() == 1 && pred.node != nullptr && pd[0] == pred.node;
            mode = want_early ? launch_mode(pred, blocked, cap_id, adjacent, mine) : 0;
            if (pin < 0) c.pinned.push_back(h);
            if (head) c.n_br = b + 1;
            add_ranges(c.br[b].rd, mine->rd, mine->n_rd);
            add_ranges(c.br[b].wr, mine->wr, mine->n_wr);
            g_branch = b; g_branch_head = head && b > 0; g_cross_branch = c.last >= 0 && c.last != b;
            c.last = b;
        }
    }
    if (b < 0) {
        const bool adjacent = (cap_id != 0 && n_d == 1 && t.node != nullptr && deps[0] == t.node) ||   // proven by the capture
                              (g_adjacent_hint && (cap_id == 0 || n_d == 1));                        // issued back to back by one call
        const bool blocked = t.h == h || (in_chain && contains(c.pinned, h));   // (a chain's tips are direct predecessors)
        mode = want_early ? launch_mode(t, blocked, cap_id, adjacent, mine) : 0;
        c.active = false;
    }
    StreamTail now;
    if (mine != nullptr) now = *mine;
    now.h = h; now.cap_id = cap_id; now.node = nullptr; now.pure_step = false;
    r.tail = now;
    if (g_branch >= 0) c.br[g_branch].tail = now;
    return mode;
}

// after a launch inside a capture: remember its graph node, so that the next launch can prove it is adjacent
static void note_launched(cudaStream_t s, bool pure_step) {
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    unsigned long long cap_id = 0;
    const cudaGraphNode_t* deps = nullptr;
    size_t n_deps = 0;
    // (eager launches have no graph node: the driver call is only made while the stream is being captured)
    if (g_capturing && cudaStreamGetCaptureInfo(s, &cap, &cap_id, nullptr, &deps, &n_deps) != cudaSuccess) { cudaGetLastError(); return; }
    std::lock_guard<std::mutex> lk(g_order_mu);
    auto it = g_streams.find(s);
    if (it == g_streams.end()) return;
    StreamTail& t = it->second.tail;
    t.pure_step = pure_step;
    t.node = (cap == cudaStreamCaptureStatusActive && n_deps == 1) ? deps[0] : nullptr;
    if (g_branch >= 0 && it->second.chain.active) {
        StreamTail& bt = it->second.chain.br[g_branch].tail;
        bt.pure_step = t.pure_step; bt.node = t.node;
    }
}

// after the last launch that claim_stream placed on a branch (the step and the queued-reset kernel behind it): the stream
// depends on every branch's tip again
static cudaError_t join_branches(cudaStream_t s) {
    if (g_branch < 0) return cudaSuccess;
    g_branch = -1;
    std::lock_guard<std::mutex> lk(g_order_mu);
    auto it = g_streams.find(s);
    if (it == g_streams.end() || !it->second.chain.active) return cudaSuccess;
    Chain& c = it->second.chain;
    c.left.clear();
    for (int b = 0; b < c.n_br; b++) {
        if (c.br[b].tail.node == nullptr) { c.active = false; return cudaErrorStreamCaptureInvalidated; }
        c.left.push_back(c.br[b].tail.node);
    }
    const cudaError_t e = cudaStreamUpdateCaptureDependencies(s, c.left.data(), c.left.size(), cudaStreamSetCaptureDependencies);
    if (e != cudaSuccess) c.active = false;
    return e;
}

static void forget_handle(ngw_handle* h) {
    std::lock_guard<std::mutex> lk(g_order_mu);
    for (auto& kv : g_streams) {
        const Chain& c = kv.second.chain;
        if (kv.second.tail.h == h || contains(c.pinned, h) || contains(c.base_block, h)) {
            kv.second.tail.h = nullptr;
            kv.second.chain.active = false;
        }
    }
}

static int before_device_call(ngw_handle* h, cudaStream_t s) {
    if (h->host_dirty) {
        if (cudaStreamSynchronize(h->hs) != cudaSuccess) { cudaGetLastError(); }
        h->host_dirty = false;
    }
    h->last_dev_stream = s;
    h->dev_dirty = true;
    return 0;
}

// for the entry points that write state with plain kernels / copies (no programmatic launch): the next step on this
// stream must not load early if it belongs to the same handle
static void note_state_writer(ngw_handle* h, cudaStream_t s) { claim_stream(h, s, false); }

extern "C" {

const char* ngw_last_error(void) { return g_err.c_str(); }
int ngw_abi_version(void) { return NGW_ABI_VERSION; }

void ngw_destroy(ngw_handle* h) {
    if (!h) return;
    forget_handle(h);
    cudaSetDevice(h->device);
    if (h->hs) cudaStreamSynchronize(h->hs);
    for (auto p : h->d_luts) cudaFree(p);
    cudaFree(h->d_cfgs); cudaFree(h->map); cudaFree(h->pose); cudaFree(h->inv); cudaFree(h->cfg_id);
    cudaFree(h->episode); cudaFree(h->ep_len); cudaFree(h->err); cudaFree(h->stats); cudaFree(h->zero_byte); cudaFree(h->reset_list); cudaFree(h->reset_ctl);
    cudaFree(h->mt_key); cudaFree(h->mt_pos);
    cudaFree(h->h_actions); cudaFree(h->h_obs);   // reward / step_cost / done / result staging lives in h_obs's block
    if (h->hs) cudaStreamDestroy(h->hs);
    if (h->ev_dev) cudaEventDestroy(h->ev_dev);
    delete h;
}

static int create_init(ngw_handle* h, const ngw_config* cfgs, int32_t n_cfgs, int64_t n_envs, int32_t map_size,
                       int32_t device, int64_t first_env_gid, uint64_t seed, const cudaDeviceProp& prop);

int ngw_create(ngw_handle** out, const ngw_config* cfgs, int32_t n_cfgs, int64_t n_envs, int32_t map_size,
               int32_t device, int64_t first_env_gid, uint64_t seed) {
    if (!out || !cfgs || n_cfgs < 1 || n_cfgs > 255) return fail("ngw_create: need 1..255 configs");
    if (n_envs < 1) return fail("ngw_create: n_envs must be >= 1");
    if (map_size < 5 || map_size > NGW_MAX_MAP_SIZE) return fail("ngw_create: map_size out of range");
    CK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return fail("ngw_create: this library is built for sm_100a (B200) only");
    ngw_handle* h = new ngw_handle();
    h->device = device;
    if (create_init(h, cfgs, n_cfgs, n_envs, map_size, device, first_env_gid, seed, prop)) {
        std::string why = g_err;                    // ngw_destroy must not clobber the reason
        ngw_destroy(h);
        g_err = why;
        return 1;
    }
    *out = h;
    return 0;
}

// compass directions (d_row, d_col) of the line-gather lidar, see ngw_device.cuh
static const int kCompass[8][2] = {{1, 0}, {1, 1}, {0, 1}, {-1, 1}, {-1, 0}, {-1, -1}, {0, -1}, {1, -1}};

// Host beam LUT (d_row, d_col per facing / beam / sample, generated with the reference's own NumPy expression) ->
// device tables.  Returns the path the kernels will take: 0 no lidar, 1 generic LUT walk, 2 factorised pointer walk,
// 3 line gather.  `lin` (optional) receives the int16 linear-offset LUT of the generic path.
static int build_lidar_tables(const ngw_config& c, int map_size, LidarDev& ld, std::vector<int16_t>* lin) {
    memset(&ld, 0, sizeof(ld));
    const int B = c.n_beams, K = c.max_range;
    if (B <= 0 || c.beam_lut == nullptr) return 0;
    auto at = [&](int f, int b, int k, int j) { return (int)c.beam_lut[((f * B + b) * K + k) * 2 + j]; };
    bool fast = (B == 8 && K >= 1 && K <= NGW_MAX_RANGE);
    if (fast) {
        for (int par = 0; par < 2 && fast; par++)
            for (int k = 0; k < K && fast; k++) {
                int dr = abs(at(0, par, k, 0)), dcol = abs(at(0, par, k, 1));
                int d = dr > dcol ? dr : dcol;
                if (d > 255) fast = false;
                ld.disp[par][k] = (uint8_t)d;
            }
        for (int f = 0; f < 4 && fast; f++)
            for (int b = 0; b < 8 && fast; b++) {
                int ur = at(f, b, 0, 0), uc = at(f, b, 0, 1);
                if (abs(ur) > 1 || abs(uc) > 1 || (ur == 0 && uc == 0)) { fast = false; break; }
                ld.unit[f][b] = (int16_t)(ur * map_size + uc);
                for (int k = 0; k < K; k++) {
                    int d = ld.disp[b & 1][k];
                    if (at(f, b, k, 0) != ur * d || at(f, b, k, 1) != uc * d) { fast = false; break; }
                }
            }
    }
    // line gather: beam b of facing f looks along compass direction (b + rot[f]) & 7 with rot even, axis beams travel
    // k cells at sample k, diagonal beams start at 1 cell and never skip a cell
    bool lines = fast && K <= 255;
    if (lines) {
        for (int k = 0; k < K && lines; k++) {
            if (ld.disp[0][k] != k + 1) lines = false;
            int prev = k ? ld.disp[1][k - 1] : 0;
            if (ld.disp[1][k] != prev && ld.disp[1][k] != prev + 1) lines = false;
        }
        if (lines && ld.disp[1][0] != 1) lines = false;
        if (lines && ld.disp[1][K - 1] > NGW_MAX_MAP_SIZE) lines = false;
        for (int f = 0; f < 4 && lines; f++) {
            int rot = -1;
            for (int a = 0; a < 8; a++)
                if (at(f, 0, 0, 0) == kCompass[a][0] && at(f, 0, 0, 1) == kCompass[a][1]) rot = a;
            if (rot < 0 || (rot & 1)) { lines = false; break; }
            for (int b = 0; b < 8; b++) {
                const int a = (b + rot) & 7;
                if (at(f, b, 0, 0) != kCompass[a][0] || at(f, b, 0, 1) != kCompass[a][1]) lines = false;
            }
            ld.rot[f] = (uint8_t)rot;
        }
        if (lines)
            for (int k = K - 1; k >= 0; k--) ld.firstk[ld.disp[1][k] - 1] = (uint8_t)(k + 1);   // first sample reaching cell d
    }
    if (!lines) { memset(ld.firstk, 0, sizeof(ld.firstk)); memset(ld.rot, 0, sizeof(ld.rot)); }
    ld.fast = fast ? 1 : 0;
    ld.lines = lines ? 1 : 0;
    if (!fast && lin) {
        int n = 4 * B * K;
        lin->resize(n);
        for (int j = 0; j < n; j++) (*lin)[j] = (int16_t)(c.beam_lut[2 * j] * map_size + c.beam_lut[2 * j + 1]);
    }
    return lines ? 3 : (fast ? 2 : 1);
}

int ngw_lidar_path(const ngw_config* cfg, int32_t map_size) {
    if (!cfg) return -1;
    LidarDev ld;
    return build_lidar_tables(*cfg, map_size, ld, nullptr);
}

static int obs_row_bytes_of(const ngw_handle* h, int format) {
    int best = 0;
    for (const DevConfig& dc : h->h_cfgs) {
        const ngw_config& c = dc.c;
        if (c.n_beams <= 0) continue;
        const int b = obs_tail_offset(format, c.n_lidar_items, c.n_beams) + 4 * c.n_inv_obs;
        if (b > best) best = b;
    }
    return best;
}

// Function attributes of every kernel, on the current device (the handle's: create_init runs after cudaSetDevice).
static int set_kernel_attributes() {
#define NGW_SMEM_ATTR(K) CK(cudaFuncSetAttribute(K, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024))
#define NGW_SMEM_ATTR4(K, ...) NGW_SMEM_ATTR((K<0, __VA_ARGS__>)); NGW_SMEM_ATTR((K<1, __VA_ARGS__>)); \
                               NGW_SMEM_ATTR((K<4, __VA_ARGS__>)); NGW_SMEM_ATTR((K<16, __VA_ARGS__>))
    NGW_SMEM_ATTR4(step1_kernel, true, true); NGW_SMEM_ATTR4(step1_kernel, true, false); NGW_SMEM_ATTR4(step1_kernel, false, false);
    NGW_SMEM_ATTR4(step1w_kernel, 8); NGW_SMEM_ATTR4(step1w_kernel, 16);
#undef NGW_SMEM_ATTR4
#undef NGW_SMEM_ATTR
    // the queued-reset kernel shares SMs with the next handle's step CTAs: both must want the same (maximal) shared-memory
    // carve-out, or the SM would have to drain before it can be reconfigured
    CK(cudaFuncSetAttribute(reset_list_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    // the numpy reset stream's candidate lists (ms^2 uint16 per warp) take both reset kernels past the 48 KB a launch gets
    // without opting in on grids above ~58x58; the Philox plans are below it and do not change
    CK(cudaFuncSetAttribute(reset_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024 - (int)sizeof(ResetScratch) * NGW_RESET_WARPS));
    CK(cudaFuncSetAttribute(reset_list_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    return ngw_rollout_set_attributes();              // ngw_rollout.cu
}

static int create_init(ngw_handle* h, const ngw_config* cfgs, int32_t n_cfgs, int64_t n_envs, int32_t map_size,
                       int32_t device, int64_t first_env_gid, uint64_t seed, const cudaDeviceProp& prop) {
    h->device = device; h->n = n_envs; h->np = (n_envs + 31) / 32 * 32; h->first_gid = first_env_gid; h->seed = seed;
    h->ms = map_size; h->cells = map_size * map_size; h->n_cfgs = n_cfgs;
    h->concurrent = getenv("NGW_NO_CONCURRENT") == nullptr;
    // test knob: key ties.  It reaches ngw_reset and the one-step auto-resets; the rollouts' in-place resets keep every key bit
    if (const char* km = getenv("NGW_DEBUG_KEY_MASK")) h->key_mask = (uint32_t)strtoul(km, nullptr, 0);
    for (int i = 0; i < n_cfgs; i++) {
        const ngw_config& c = cfgs[i];
        if (c.n_items < 1 || c.n_items > NGW_MAX_ITEMS || c.n_actions < 0 || c.n_actions > NGW_MAX_ACTIONS ||
            c.n_recipes > NGW_MAX_RECIPES || c.n_place > NGW_MAX_PLACE || c.n_reset_ops > NGW_MAX_RESET_OPS ||
            c.n_beams < 0 || c.max_range < 0 || c.n_beams * c.max_range > 4096) {
            return fail("ngw_create: config " + std::to_string(i) + " out of range");
        }
        if (c.n_items > h->inv_stride) h->inv_stride = c.n_items;
        int d = c.n_beams > 0 ? c.n_lidar_items * c.n_beams + c.n_inv_obs : 0;
        if (d > h->obs_dim) h->obs_dim = d;
        if (c.n_beams > 0 && c.beam_lut == nullptr) return fail("ngw_create: lidar config without beam_lut");
    }
    h->h_cfgs.resize(n_cfgs);
    for (int i = 0; i < n_cfgs; i++) {
        DevConfig& dc = h->h_cfgs[i];
        memset(&dc, 0, sizeof(dc));
        dc.c = cfgs[i];
        std::vector<int16_t> lin;
        build_lidar_tables(cfgs[i], map_size, dc.lidar, &lin);
        int16_t* d_lut = nullptr;
        if (!lin.empty()) {
            CK(cudaMalloc(&d_lut, lin.size() * sizeof(int16_t)));
            CK(cudaMemcpy(d_lut, lin.data(), lin.size() * sizeof(int16_t), cudaMemcpyHostToDevice));
            h->d_luts.push_back(d_lut);
        }
        dc.lidar.lut = d_lut;
        dc.c.beam_lut = nullptr;
        // the observation's inventory tail as an id range (the usual case: ids follow the sorted names)
        dc.lidar.tail_first = dc.c.n_inv_obs > 0 ? (int)dc.c.inv_obs_item[0] : -1;
        for (int j = 0; j < dc.c.n_inv_obs; j++)
            if ((int)dc.c.inv_obs_item[j] != dc.lidar.tail_first + j) dc.lidar.tail_first = -1;
    }
    h->lidar_uniform = n_cfgs > 1;
    for (int i = 1; i < n_cfgs; i++) {
        const LidarDev &a = h->h_cfgs[0].lidar, &b = h->h_cfgs[i].lidar;
        if (!a.fast || !b.fast || (a.lines != 0) != (b.lines != 0) || h->h_cfgs[0].c.max_range != h->h_cfgs[i].c.max_range ||
            memcmp(a.unit, b.unit, sizeof(a.unit)) != 0 || memcmp(a.disp, b.disp, sizeof(a.disp)) != 0)
            h->lidar_uniform = false;
    }
    CK(cudaMalloc(&h->d_cfgs, sizeof(DevConfig) * n_cfgs));
    CK(cudaMemcpy(h->d_cfgs, h->h_cfgs.data(), sizeof(DevConfig) * n_cfgs, cudaMemcpyHostToDevice));
    // state
    CK(cudaMalloc(&h->map, (size_t)h->np * h->cells));
    CK(cudaMalloc(&h->pose, (size_t)h->np * 4));
    CK(cudaMalloc(&h->inv, (size_t)h->np * h->inv_stride * 4));
    CK(cudaMalloc(&h->cfg_id, (size_t)h->np));
    CK(cudaMalloc(&h->episode, (size_t)h->np * 4));
    CK(cudaMalloc(&h->ep_len, (size_t)h->np * 4));
    CK(cudaMalloc(&h->err, (size_t)h->np * 4));
    CK(cudaMalloc(&h->stats, sizeof(double) * NGW_STAT_SLOTS * NGW_STAT_COUNT));
    CK(cudaMalloc(&h->reset_list, (size_t)h->np * 4));
    CK(cudaMalloc(&h->reset_ctl, 16));
    CK(cudaMemset(h->reset_ctl, 0, 16));
    h->sm_count = prop.multiProcessorCount;
    CK(cudaMalloc(&h->zero_byte, 16));
    CK(cudaMemset(h->zero_byte, 0, 16));
    CK(cudaMemset(h->map, 0, (size_t)h->np * h->cells));
    CK(cudaMemset(h->pose, 0, (size_t)h->np * 4));
    CK(cudaMemset(h->inv, 0, (size_t)h->np * h->inv_stride * 4));
    CK(cudaMemset(h->cfg_id, 0, (size_t)h->np));
    CK(cudaMemset(h->episode, 0, (size_t)h->np * 4));
    CK(cudaMemset(h->ep_len, 0, (size_t)h->np * 4));
    CK(cudaMemset(h->err, 0, (size_t)h->np * 4));
    CK(cudaMemset(h->stats, 0, sizeof(double) * NGW_STAT_SLOTS * NGW_STAT_COUNT));
    // bytes of one 32-env tile of each array
    h->map_bytes = 32 * h->cells;                       // multiple of 32
    h->inv_bytes = 128 * h->inv_stride;
    h->obs_format = NGW_OBS_I32;
    h->obs_row_bytes = obs_row_bytes_of(h, NGW_OBS_I32);
    h->obs_bytes = 32 * h->obs_row_bytes;
    const int one_tile = NGW_SMEM_HDR + 512 + 1280 + h->map_bytes + h->inv_bytes + 128 * h->obs_dim;
    if (one_tile > 227 * 1024) return fail("ngw_create: map too large for shared memory");
    // G warps share one tile (the first two split the step by action class, all G cast the lidar lines): 2 for small
    // grids, 4 when shared memory limits the tiles per SM to a few
    int tiles_per_sm = (227 * 1024) / (one_tile + 1024);
    int warps = tiles_per_sm >= 6 ? 2 : 4;
    if (n_cfgs > 1 && warps == 2) warps = 1;      // mixed batches: a second warp repeats the per-lane config reads (C4 129 vs 139 us)
    h->warps = warps;
    // line-gather lidar with one geometry for the whole batch (the common case): the kernel skips the per-lane dispatch
    h->lidar_mode = 1;
    for (int i = 0; i < n_cfgs; i++) {
        const DevConfig& dc = h->h_cfgs[i];
        if (dc.c.n_beams <= 0 || !dc.lidar.lines) h->lidar_mode = 0;
    }
    if (n_cfgs > 1 && !h->lidar_uniform) h->lidar_mode = 0;
    if (map_size > 32) h->lidar_mode = 0;           // large grids: pointer-walking beams (lidar_observe decides per lane)
    return set_kernel_attributes();
}

int ngw_state(ngw_handle* h, ngw_state_view* o) {
    if (!h || !o) return fail("ngw_state: null");
    o->map = h->map; o->pose = reinterpret_cast<uint8_t*>(h->pose); o->inventory = h->inv; o->cfg_id = h->cfg_id;
    o->episode = h->episode; o->ep_len = h->ep_len; o->error_flags = h->err;
    o->inv_stride = h->inv_stride; o->obs_dim = h->obs_dim; o->n_envs = h->n; o->n_envs_padded = h->np;
    o->map_size = h->ms; o->n_configs = h->n_cfgs;
    o->obs_format = h->obs_format; o->obs_row_bytes = h->obs_row_bytes;
    return 0;
}

int ngw_set_obs_format(ngw_handle* h, int32_t format) {
    if (!h) return fail("null handle");
    if (format != NGW_OBS_I32 && format != NGW_OBS_U8 && format != NGW_OBS_HITS)
        return fail("ngw_set_obs_format: unknown format");
    if (format != NGW_OBS_I32)                     // both narrow layouts store a range in one byte
        for (const DevConfig& dc : h->h_cfgs)
            if (dc.c.max_range > 255) return fail("ngw_set_obs_format: max_range does not fit a byte");
    if (h->host_dirty) { cudaStreamSynchronize(h->hs); h->host_dirty = false; }
    h->obs_format = format;
    h->obs_row_bytes = obs_row_bytes_of(h, format);
    h->obs_bytes = 32 * h->obs_row_bytes;
    return 0;
}

int ngw_set_env_configs(ngw_handle* h, const int32_t* cfg_id_dev, void* stream) {
    if (!h) return fail("null handle");
    CK(cudaSetDevice(h->device));
    before_device_call(h, (cudaStream_t)stream);
    note_state_writer(h, (cudaStream_t)stream);
    int blocks = (int)((h->n + 255) / 256);
    set_cfg_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(cfg_id_dev, h->cfg_id, h->n, h->n_cfgs, h->err);
    h->launches++;
    CK(cudaGetLastError());
    return 0;
}

int ngw_load_state(ngw_handle* h, const int8_t* map, const uint8_t* pose, const int32_t* inventory, int64_t first,
                   int64_t count, void* stream) {
    if (!h) return fail("null handle");
    if (first < 0 || count < 0 || first + count > h->n) return fail("ngw_load_state: range outside the batch");
    CK(cudaSetDevice(h->device));
    cudaStream_t s = (cudaStream_t)stream;
    before_device_call(h, s);
    note_state_writer(h, s);
    if (map) CK(cudaMemcpyAsync(h->map + first * h->cells, map, (size_t)count * h->cells, cudaMemcpyDeviceToDevice, s));
    if (pose) CK(cudaMemcpyAsync(h->pose + first, pose, (size_t)count * 4, cudaMemcpyDeviceToDevice, s));
    if (inventory)
        CK(cudaMemcpyAsync(h->inv + first * h->inv_stride, inventory, (size_t)count * h->inv_stride * 4,
                           cudaMemcpyDeviceToDevice, s));
    CK(cudaMemsetAsync(h->ep_len + first, 0, (size_t)count * 4, s));
    return 0;
}

int ngw_export_state(ngw_handle* h, int8_t* map, uint8_t* pose, int32_t* inventory, int64_t first, int64_t count,
                     void* stream) {
    if (!h) return fail("null handle");
    if (first < 0 || count < 0 || first + count > h->n) return fail("ngw_export_state: range outside the batch");
    CK(cudaSetDevice(h->device));
    cudaStream_t s = (cudaStream_t)stream;
    before_device_call(h, s);
    // cudaMemcpyDefault: the destinations may be device or (pinned / pageable) host memory
    if (map) CK(cudaMemcpyAsync(map, h->map + first * h->cells, (size_t)count * h->cells, cudaMemcpyDefault, s));
    if (pose) CK(cudaMemcpyAsync(pose, h->pose + first, (size_t)count * 4, cudaMemcpyDefault, s));
    if (inventory)
        CK(cudaMemcpyAsync(inventory, h->inv + first * h->inv_stride, (size_t)count * h->inv_stride * 4,
                           cudaMemcpyDefault, s));
    return 0;
}

int ngw_set_reset_rng(ngw_handle* h, int32_t kind, void* stream) {
    if (!h) return fail("null handle");
    if (kind != NGW_RNG_PHILOX && kind != NGW_RNG_NUMPY) return fail("ngw_set_reset_rng: unknown generator kind");
    CK(cudaSetDevice(h->device));
    if (kind == NGW_RNG_PHILOX) {
        // (cudaFree waits for the device: no launch still reading the state can outlive it)
        if (h->mt_key) { CK(cudaFree(h->mt_key)); CK(cudaFree(h->mt_pos)); }
        h->mt_key = nullptr; h->mt_pos = nullptr;
        return 0;
    }
    if (h->first_gid < 0 || h->seed + (unsigned long long)h->first_gid + (unsigned long long)(h->n - 1) >= (1ull << 32))
        return fail("ngw_set_reset_rng: np.random.seed takes seeds below 2^32, but seed + first_env_gid + n_envs - 1 = " +
                    std::to_string(h->seed + (unsigned long long)h->first_gid + (unsigned long long)(h->n - 1)));
    if (!h->mt_key) {
        uint32_t* key = nullptr; int32_t* pos = nullptr;
        CK(cudaMalloc(&key, (size_t)h->np * NGW_MT_WORDS * 4));
        if (cudaMalloc(&pos, (size_t)h->np * 4) != cudaSuccess) {
            cudaGetLastError();
            cudaFree(key);
            return fail("ngw_set_reset_rng: out of device memory for the np.random states");
        }
        h->mt_key = key; h->mt_pos = pos;     // mt_seed_kernel writes every env's state; the padding rows are never read
    }
    cudaStream_t s = (cudaStream_t)stream;
    before_device_call(h, s);
    note_state_writer(h, s);
    mt_seed_kernel<<<(unsigned)((h->n + 127) / 128), 128, 0, s>>>(h->mt_key, h->mt_pos, h->n,
                                                                 h->seed + (unsigned long long)h->first_gid);
    h->launches++;
    CK(cudaGetLastError());
    return 0;
}

// the checks the two state copies share: a numpy-stream handle and a range inside the batch
static int rng_state_range(const ngw_handle* h, const char* who, int64_t first, int64_t count) {
    if (!h) return fail("null handle");
    if (!h->mt_key) return fail(std::string(who) + ": the handle has no np.random states (ngw_set_reset_rng(NGW_RNG_NUMPY))");
    if (first < 0 || count < 0 || first + count > h->n) return fail(std::string(who) + ": range outside the batch");
    return 0;
}

int ngw_load_rng_state(ngw_handle* h, const uint32_t* key, const int32_t* pos, int64_t first, int64_t count, void* stream) {
    if (rng_state_range(h, "ngw_load_rng_state", first, count)) return 1;
    if (count == 0) return 0;
    if (!key || !pos) return fail("ngw_load_rng_state: null key or pos");
    CK(cudaSetDevice(h->device));
    cudaStream_t s = (cudaStream_t)stream;
    // pos is checked on the host before anything is enqueued: once the stream's earlier work has written it
    std::vector<int32_t> hp((size_t)count);
    CK(cudaStreamSynchronize(s));
    CK(cudaMemcpy(hp.data(), pos, (size_t)count * 4, cudaMemcpyDeviceToHost));
    for (int64_t i = 0; i < count; i++)
        if (hp[(size_t)i] < 0 || hp[(size_t)i] > NGW_MT_WORDS)
            return fail("ngw_load_rng_state: pos[" + std::to_string(i) + "] = " + std::to_string(hp[(size_t)i]) +
                        " outside [0, 624]");
    before_device_call(h, s);
    note_state_writer(h, s);
    CK(cudaMemcpyAsync(h->mt_key + first * NGW_MT_WORDS, key, (size_t)count * NGW_MT_WORDS * 4, cudaMemcpyDeviceToDevice, s));
    CK(cudaMemcpyAsync(h->mt_pos + first, pos, (size_t)count * 4, cudaMemcpyDeviceToDevice, s));
    return 0;
}

int ngw_export_rng_state(ngw_handle* h, uint32_t* key, int32_t* pos, int64_t first, int64_t count, void* stream) {
    if (rng_state_range(h, "ngw_export_rng_state", first, count)) return 1;
    CK(cudaSetDevice(h->device));
    cudaStream_t s = (cudaStream_t)stream;
    before_device_call(h, s);
    note_state_writer(h, s);                  // ends a capture chain: the copies wait for every branch
    // cudaMemcpyDefault: the destinations may be device or (pinned / pageable) host memory
    if (key) CK(cudaMemcpyAsync(key, h->mt_key + first * NGW_MT_WORDS, (size_t)count * NGW_MT_WORDS * 4, cudaMemcpyDefault, s));
    if (pos) CK(cudaMemcpyAsync(pos, h->mt_pos + first, (size_t)count * 4, cudaMemcpyDefault, s));
    return 0;
}

static ResetParams reset_params(ngw_handle* h, const uint8_t* mask, int phase) {
    ResetParams p;
    p.dcfgs = h->d_cfgs; p.map = h->map; p.pose = h->pose; p.inv = h->inv; p.cfg_id = h->cfg_id; p.episode = h->episode;
    p.ep_len = h->ep_len; p.err = h->err; p.mask = mask; p.n_envs = h->n; p.first_gid = h->first_gid; p.seed = h->seed;
    p.ms = h->ms; p.cells = h->cells; p.inv_stride = h->inv_stride; p.phase = phase; p.zero_byte = h->zero_byte;
    p.reset_list = h->reset_list; p.reset_count = h->reset_ctl; p.done_ctas = h->reset_ctl + 1; p.obs = nullptr;
    p.final_obs = nullptr;
    p.obs_dim = h->obs_dim; p.obs_row_bytes = h->obs_row_bytes; p.obs_format = h->obs_format;
    p.key_mask = h->key_mask;
    p.mt_key = h->mt_key; p.mt_pos = h->mt_pos;
    return p;
}

int ngw_reset(ngw_handle* h, const uint8_t* mask, void* obs, void* stream) {
    if (!h) return fail("null handle");
    CK(cudaSetDevice(h->device));
    cudaStream_t s = (cudaStream_t)stream;
    before_device_call(h, s);
    note_state_writer(h, s);
    int blocks = (int)((h->n + 127) / 128);
    int rblocks = (int)((h->n + NGW_RESET_WARPS - 1) / NGW_RESET_WARPS);
    bool split = false;
    for (auto& c : h->h_cfgs) split |= c.c.reset_obs_after_ops < c.c.n_reset_ops;
    const bool want_obs = obs != nullptr && h->obs_dim > 0;
    ResetParams po = reset_params(h, mask, split ? 0 : 2);
    po.obs = static_cast<unsigned char*>(obs);
    // numpy stream: every warp's candidate list (the Philox reset needs no dynamic shared memory)
    const size_t lists = h->mt_key != nullptr ? (size_t)NGW_RESET_WARPS * 2 * h->cells : 0;
    if (!want_obs || !split) {
        reset_kernel<<<rblocks, 32 * NGW_RESET_WARPS, lists, s>>>(reset_params(h, mask, 2));
        h->launches++;
        if (want_obs) {
            observe_masked_kernel<<<blocks, 128, 0, s>>>(po);
            h->launches++;
        }
    } else {
        reset_kernel<<<rblocks, 32 * NGW_RESET_WARPS, lists, s>>>(reset_params(h, mask, 0));
        observe_masked_kernel<<<blocks, 128, 0, s>>>(po);
        reset_kernel<<<rblocks, 32 * NGW_RESET_WARPS, lists, s>>>(reset_params(h, mask, 1));
        h->launches += 3;
    }
    CK(cudaGetLastError());
    return 0;
}

static StepParams step_params(ngw_handle* h, const int32_t* actions, void* obs, float* reward, uint8_t* done,
                              float* cost, uint8_t* result, int auto_reset, int max_episode_steps, long long begin,
                              long long end) {
    StepParams p;
    memset(&p, 0, sizeof(p));
    p.dcfgs = h->d_cfgs; p.map = h->map; p.pose = h->pose; p.inv = h->inv; p.cfg_id = h->cfg_id; p.episode = h->episode;
    p.ep_len = h->ep_len; p.err = h->err; p.actions = actions;
    p.obs = h->obs_dim > 0 ? static_cast<unsigned char*>(obs) : nullptr; p.reward = reward;
    p.done = done; p.cost = cost; p.result = result; p.stats = h->stats;
    p.env_begin = begin; p.env_end = end; p.first_gid = h->first_gid; p.seed = h->seed;
    p.ms = h->ms; p.cells = h->cells; p.inv_stride = h->inv_stride; p.obs_dim = h->obs_dim;
    p.map_bytes = h->map_bytes; p.inv_bytes = h->inv_bytes; p.obs_bytes = h->obs_bytes;
    p.obs_row_bytes = h->obs_row_bytes; p.obs_format = h->obs_format;
    p.auto_reset = auto_reset; p.max_episode_steps = max_episode_steps;
    p.lidar_uniform = h->lidar_uniform ? 1 : 0;
    p.msg = h->msg; p.reset_list = h->reset_list; p.reset_count = h->reset_ctl;
    // episode-end buffers: stepping launches only (observe-only launches leave them alone; the rollouts clear them), and
    // a final observation only where there is one
    p.trunc = actions != nullptr ? h->trunc : nullptr;
    p.final_obs = actions != nullptr && p.obs != nullptr ? h->final_obs : nullptr;
    p.n_steps = 1;
    p.mt_key = h->mt_key; p.mt_pos = h->mt_pos;
    return p;
}

}  // extern "C" (templates need C++ linkage)

static bool is_multi(const StepParams& p) {
    return p.n_steps > 1 || p.random_policy || p.done_count != nullptr || p.actions_out != nullptr || p.policy_w != nullptr ||
           p.record;
}

// shared-memory row stride of a one-step kernel's observation tile (StepParams::obs_srow): rows of a multiple of 8 words
// get 16 bytes of padding
static int obs_srow(int obs_row_bytes) {
    return obs_row_bytes + (((obs_row_bytes >> 2) % 8 == 0 && obs_row_bytes > 0) ? 16 : 0);
}

// after a one-step launch: the stream's record for the next launch's independence proof, and the handle's counters
static void note_step_launched(ngw_handle* h, cudaStream_t s, const StepParams& p) {
    note_launched(s, p.actions != nullptr);
    // launches that may overlap their stream predecessor: independent of it on one branch, or on another branch
    h->concurrent_launches += (p.concurrent || g_cross_branch) ? 1 : 0;
    h->last_step_concurrent = p.concurrent != 0;
}

// caller buffers of a one-step launch (for the independence proof of this launch and of the next one)
static StreamTail launch_tail(const StepParams& p) {
    StreamTail me;
    const long long n_env = p.env_end - p.env_begin;
    auto add = [](MemRange* r, int& n, const void* ptr, size_t bytes) {
        if (ptr != nullptr && bytes > 0) { r[n].lo = (uintptr_t)ptr; r[n].hi = (uintptr_t)ptr + bytes; n++; }
    };
    add(me.rd, me.n_rd, p.actions, (size_t)n_env * 4);
    add(me.wr, me.n_wr, p.obs, (size_t)n_env * p.obs_row_bytes);
    add(me.wr, me.n_wr, p.reward, (size_t)n_env * 4); add(me.wr, me.n_wr, p.cost, (size_t)n_env * 4);
    add(me.wr, me.n_wr, p.done, (size_t)n_env); add(me.wr, me.n_wr, p.result, (size_t)n_env);
    add(me.wr, me.n_wr, p.msg, (size_t)n_env * 2);
    // (the queued-reset kernel behind the step writes final_obs: the step's record covers it, see launch_step)
    add(me.wr, me.n_wr, p.trunc, (size_t)n_env); add(me.wr, me.n_wr, p.final_obs, (size_t)n_env * p.obs_row_bytes);
    return me;
}

// Which one-step launches may join a capture chain's branches: stepping launches of ONE wave.  Launches of several waves
// keep the two-deep chain: on the same B200 as kBranches, branching them too moved C3 23.2 -> 21.4 us per step but C5
// (auto-reset, map 40) 244 -> 267 us, and C4 not at all (96.9 / 97.2).
static bool branchable(const StepParams& p, bool one_wave) { return p.actions != nullptr && one_wave; }

// one-step launches (ngw_step / ngw_step_host / ngw_observe): several tile groups per CTA
template <int NC>
static cudaError_t launch_step1_nc(ngw_handle* h, StepParams p, cudaStream_t s) {
    // ---- shared-memory plan: CTA header | lidar tables | tiles_per_cta x (group header | grid | inventory | observation)
    p.off_luts = NGW_CTA_HDR;
    p.off_groups = p.off_luts + lut_bytes<NC>();
    p.obs_srow = obs_srow(p.obs_row_bytes);
    p.group_bytes = (NGW_GROUP_HDR + p.map_bytes + p.inv_bytes + 32 * p.obs_srow + 127) & ~127;
    // alias plan (one tile per CTA, see step1_kernel<.., kAlias>): the observation tile shares the rows' shared memory
    bool alias = true;
    for (const DevConfig& dc : h->h_cfgs)
        if (dc.c.n_inv_obs > NGW_REGSINK_TAIL || (dc.c.n_beams > 0 && !dc.lidar.lines && !dc.lidar.fast)) alias = false;
    const int alias_bytes = (NGW_GROUP_HDR + ((p.map_bytes + p.inv_bytes) > 32 * p.obs_srow ? (p.map_bytes + p.inv_bytes) : 32 * p.obs_srow) + 127) & ~127;
    const int G = h->warps;
    p.g_shift = G == 4 ? 2 : (G == 2 ? 1 : 0);
    const long long tiles = (p.env_end - p.env_begin + 31) / 32;
    // Tile groups per CTA.  A launch that fits the GPU in ONE wave (C2: 2048 tiles, 14 per SM) is bound by launch and
    // phase latency: an empty launch of 2048 one-tile CTAs costs 2.5 us, of 293 seven-tile CTAs 0.7 us — so the tiles are
    // packed into two CTAs per SM.  A launch of several waves runs one tile per CTA: small CTAs retire independently,
    // which staggers the load / compute / store phases of neighbouring tiles (C3 28.5 vs 31.7 us).
    const long long per_sm = (227 * 1024 - p.off_groups) / p.group_bytes;
    int C = 1;
    if (tiles <= per_sm * h->sm_count && per_sm >= 4) {
        C = (int)((tiles + 2 * h->sm_count - 1) / (2 * h->sm_count));
        const int c_cap = (int)((113 * 1024 - p.off_groups) / p.group_bytes);
        if (C > c_cap) C = c_cap;
        if (C > 512 / (32 * G)) C = 512 / (32 * G);
    }
    if (C > 15) C = 15;
    if (C > 512 / (32 * G)) C = 512 / (32 * G);
    while (C > 1 && (size_t)p.off_groups + (size_t)C * p.group_bytes > 227 * 1024) C--;
    if (C < 1) C = 1;
    if (C > tiles) C = (int)tiles;
    alias = alias && C == 1;
    if (alias) p.group_bytes = alias_bytes;
    p.tiles_per_cta = C;
    p.n_tiles = (int)tiles;
    p.lidar_mode = h->lidar_mode;
    // state loads before griddepcontrol.wait when the stream's previous state writer is another handle (observe-only
    // launches write no state, but they are ordered like steps: they read it)
    // only for one-wave launches: with several waves the loads of later waves never wait anyway, and issuing them ahead
    // of the tile's zero-fill measured 4 % slower (C4 122 vs 127 us)
    const StreamTail me = launch_tail(p);
    const int mode = claim_stream(h, s, true, &me, branchable(p, tiles <= per_sm * h->sm_count));
    // independent of the predecessor (see claim_stream): no thread waits for it except the gate CTA (block 0)
    p.concurrent = (mode == 2 && h->concurrent && p.actions != nullptr) ? 1 : 0;
    p.early_state = (p.concurrent || (mode >= 1 && C > 1)) ? 1 : 0;
    const size_t smem = (size_t)p.off_groups + (size_t)C * p.group_bytes;
    const dim3 grid((unsigned)((tiles + C - 1) / C) + (p.concurrent ? 1u : 0u)), block(32 * G * C);
    cudaError_t e;
    if (alias) e = launch_tiles<NC>(step1_kernel<NC, true, true>, h, p, grid, block, smem, s);
    else if (C == 1) e = launch_tiles<NC>(step1_kernel<NC, true, false>, h, p, grid, block, smem, s);
    else e = launch_tiles<NC>(step1_kernel<NC, false, false>, h, p, grid, block, smem, s);
    if (e == cudaSuccess) note_step_launched(h, s, p);
    return e;
}

// one-step launches in the warp-per-tile shape (step1w_kernel): returns cudaErrorNotSupported when the launch does not
// qualify and the caller should take the tile-group kernel
template <int NC>
static cudaError_t launch_step1w_nc(ngw_handle* h, StepParams p, cudaStream_t s) {
    if (h->obs_dim > 0 && h->lidar_mode != 1) return cudaErrorNotSupported;     // needs the line-gather lidar (register sink)
    int max_tail = 0;
    for (const DevConfig& dc : h->h_cfgs) max_tail = dc.c.n_inv_obs > max_tail ? dc.c.n_inv_obs : max_tail;
    if (max_tail > NGW_REGSINK_TAIL) return cudaErrorNotSupported;
    p.off_luts = NGW_WCTA_HDR;
    p.off_groups = p.off_luts + lut_bytes<NC>();
    p.obs_srow = obs_srow(p.obs_row_bytes);
    const int in_bytes = p.map_bytes + p.inv_bytes, obs_tile = p.obs ? 32 * p.obs_srow : 0;
    p.group_bytes = (NGW_WTILE_HDR + (in_bytes > obs_tile ? in_bytes : obs_tile) + 127) & ~127;
    const long long tiles = (p.env_end - p.env_begin + 31) / 32;
    // half an SM per launch: two CTAs (of this launch and the next) share an SM's 228 KB, 1 KB of each is the system's
    int c_cap = (int)((115712 - p.off_groups) / p.group_bytes);
    if (c_cap > 15) c_cap = 15;                     // 15 tile warps + the gate warp = 512 threads
    if (c_cap < 1) return cudaErrorNotSupported;
    const StreamTail me = launch_tail(p);
    const bool one_wave = tiles <= (long long)c_cap * h->sm_count;
    const int mode = claim_stream(h, s, true, &me, branchable(p, one_wave));
    p.early_state = mode >= 1 ? 1 : 0;
    // (one-wave launches overlap whole; with several waves the next launch fills the SMs as the last wave drains)
    p.concurrent = (mode == 2 && h->concurrent && p.actions != nullptr) ? 1 : 0;
    // Tiles per CTA (r02_sweep16, 29..31).  One wave, waiting for the predecessor: one CTA per SM (C2 7.3 us; two
    // 7-tile CTAs: 8.5).  One wave, overlapped: two CTAs per SM and launch, of which THREE fit an SM — one and a half
    // launches resident: C2 5.68 us vs 5.89 with 14 tiles per CTA, and 5.89 again when a slimmer header lets four
    // 7-tile CTAs in.  Several waves: 8 (C3 19.5 / 20.3 / 20.4 us with 8 / 4 / 6, C4 98.6 / 99.9 / 99.7; odd counts
    // leave partial CTAs).
    int C;
    if (!one_wave) C = 8;
    else if (p.concurrent || g_branch_head || (g_first_in_capture && h->concurrent && p.actions != nullptr))
        C = (int)((tiles + 2 * h->sm_count - 1) / (2 * h->sm_count));   // (a capture's or a branch's first launch waits, but its successor overlaps it)
    else C = (int)((tiles + h->sm_count - 1) / h->sm_count);
    if (C < 1) C = 1;
    if (C > c_cap) C = c_cap;
    if (C > tiles) C = (int)tiles;
    p.tiles_per_cta = C;
    p.n_tiles = (int)tiles;
    p.lidar_mode = h->lidar_mode;
    const size_t smem = (size_t)p.off_groups + (size_t)C * p.group_bytes;
    const dim3 grid((unsigned)((tiles + C - 1) / C)), block(32 * (C + 1));
    cudaError_t e;
    if (max_tail <= 8) e = launch_tiles<NC>(step1w_kernel<NC, 8>, h, p, grid, block, smem, s);
    else e = launch_tiles<NC>(step1w_kernel<NC, 16>, h, p, grid, block, smem, s);
    if (e == cudaSuccess) note_step_launched(h, s, p);
    return e;
}

// one-step launches: the warp-per-tile shape where it qualifies, else the tile-group kernel
template <int NC>
static cudaError_t launch_one_step(ngw_handle* h, const StepParams& p, cudaStream_t s) {
    const cudaError_t e = launch_step1w_nc<NC>(h, p, s);
    return e == cudaErrorNotSupported ? launch_step1_nc<NC>(h, p, s) : e;
}

static const int kResetCtasPerSmOverlapped = 1;    // queued-reset grid behind an overlapped step, see launch_step

static int launch_step_on_branch(ngw_handle* h, const StepParams& p, cudaStream_t s);

static int launch_step(ngw_handle* h, const StepParams& p, cudaStream_t s) {
    const int rc = launch_step_on_branch(h, p, s);
    const cudaError_t e = join_branches(s);             // (no-op unless claim_stream placed the step on a branch)
    if (rc == 0 && e != cudaSuccess) return fail(std::string("rejoining the capture branches: ") + cudaGetErrorString(e));
    return rc;
}

// the step and the queued-reset kernel behind it: on the branch claim_stream chose for the step, if any
static int launch_step_on_branch(ngw_handle* h, const StepParams& p, cudaStream_t s) {
    if (p.env_end <= p.env_begin) return 0;
    const int nc = h->n_cfgs;
    cudaError_t e;
    if (is_multi(p)) e = ngw_launch_rollout(h, p, s);   // ngw_rollout.cu
    else if (nc == 0 || nc > 16) e = launch_one_step<0>(h, p, s);
    else if (nc == 1) e = launch_one_step<1>(h, p, s);
    else if (nc <= 4) e = launch_one_step<4>(h, p, s);
    else e = launch_one_step<16>(h, p, s);
    if (e != cudaSuccess) return fail(std::string("step kernel launch: ") + cudaGetErrorString(e));
    h->launches++;
    if (p.actions != nullptr && p.auto_reset && !is_multi(p)) {     // regenerate the episodes the step kernel queued
        ResetParams rp = reset_params(h, nullptr, 2);
        rp.obs = p.obs;
        rp.final_obs = p.final_obs;
        // Grid: alone, four CTAs per SM regenerate the queue fastest (C5: ~2000 envs in 52 us).  When this step overlapped
        // its predecessor — rotating handles inside a capture — the NEXT handle's step will overlap this kernel: then ONE
        // CTA per SM (11 KB, 16 K registers) fits next to that step's full set of CTAs and the resets hide behind it.
        const int rl_ctas = h->sm_count * (h->last_step_concurrent ? kResetCtasPerSmOverlapped : 4);
        cudaLaunchConfig_t lc;
        memset(&lc, 0, sizeof(lc));
        lc.gridDim = dim3((unsigned)rl_ctas); lc.blockDim = dim3(32 * NGW_RESET_WARPS);
        lc.dynamicSmemBytes = NGW_RESET_WARPS * reset_list_scratch_bytes(h->cells, h->mt_key != nullptr);
        lc.stream = s;
        // a PLAIN launch: it starts once the step has completed.  (Launched programmatically behind an overlapped step it
        // could start under that step's tail, but that measured no faster — 250.2 vs 250.7 us on C5.)
        CK(cudaLaunchKernelEx(&lc, reset_list_kernel, rp));
        h->launches++;
        CK(cudaGetLastError());
        // a plain launch: it starts once the step has completed and lets the stream's next launch start right away
        // (griddepcontrol.launch_dependents at its top) — the next handle's step may overlap it
        note_launched(s, true);
    }
    return 0;
}

extern "C" {

int ngw_step(ngw_handle* h, const int32_t* actions, void* obs, float* reward, uint8_t* done, float* step_cost,
             uint8_t* result, int32_t auto_reset, int32_t max_episode_steps, void* stream) {
    if (!h) return fail("null handle");
    if (!actions || !reward || !done || !step_cost || !result) return fail("ngw_step: null output/action pointer");
    if (h->obs_dim > 0 && obs && ((uintptr_t)obs & 15)) return fail("ngw_step: obs must be 16-byte aligned");
    CK(cudaSetDevice(h->device));
    before_device_call(h, (cudaStream_t)stream);
    return launch_step(h, step_params(h, actions, obs, reward, done, step_cost, result, auto_reset, max_episode_steps,
                                      0, h->n), (cudaStream_t)stream);
}

int ngw_step_many(const ngw_step_item* items, int32_t n_items, int32_t auto_reset, int32_t max_episode_steps, void* stream) {
    if (!items || n_items < 0) return fail("ngw_step_many: null items");
    for (int i = 0; i < n_items; i++) {
        const ngw_step_item& it = items[i];
        if (!it.h) return fail("ngw_step_many: null handle");
        if (!it.actions || !it.reward || !it.done || !it.step_cost || !it.result) return fail("ngw_step_many: null output/action pointer");
        if (it.h->obs_dim > 0 && it.obs && ((uintptr_t)it.obs & 15)) return fail("ngw_step_many: obs must be 16-byte aligned");
        if (it.h->device != items[0].h->device) return fail("ngw_step_many: all handles must live on one device");
    }
    if (n_items == 0) return 0;
    CK(cudaSetDevice(items[0].h->device));
    int rc = 0;
    for (int i = 0; i < n_items && rc == 0; i++) {
        const ngw_step_item& it = items[i];
        before_device_call(it.h, (cudaStream_t)stream);
        g_adjacent_hint = i > 0;                        // nothing was enqueued between item i - 1's launches and this one
        rc = launch_step(it.h, step_params(it.h, it.actions, it.obs, it.reward, it.done, it.step_cost, it.result, auto_reset,
                                           max_episode_steps, 0, it.h->n), (cudaStream_t)stream);
        g_adjacent_hint = false;
    }
    return rc;
}

// a rollout with the handle's record (if one is set; the launcher passes it to the recording kernel); fails when the record
// holds fewer than n_steps steps
static int attach_record(const ngw_handle* h, StepParams& p, int32_t n_steps, const char* who) {
    if (!h->rec_on) return 0;
    if (n_steps > h->rec.max_steps)
        return fail(std::string(who) + ": n_steps " + std::to_string(n_steps) + " > the rollout record's max_steps " +
                    std::to_string(h->rec.max_steps));
    p.record = 1;
    return ngw_rollout_record_fits(h, p);
}

int ngw_rollout(ngw_handle* h, const int32_t* actions, int32_t n_steps, uint64_t policy_seed, void* obs,
                float* reward_sum, float* cost_sum, int32_t* done_count, uint8_t* last_done, uint8_t* last_result,
                int32_t* actions_out, int32_t auto_reset, int32_t max_episode_steps, void* stream) {
    if (!h) return fail("null handle");
    if (n_steps < 1) return fail("ngw_rollout: n_steps must be >= 1");
    if (!reward_sum || !cost_sum || !last_done || !last_result) return fail("ngw_rollout: null output pointer");
    if (h->obs_dim > 0 && obs && ((uintptr_t)obs & 15)) return fail("ngw_rollout: obs must be 16-byte aligned");
    // any non-null pointer marks "stepping"; with the random policy it is never dereferenced
    const int32_t* act = actions ? actions : reinterpret_cast<const int32_t*>(h->zero_byte);
    StepParams p = step_params(h, act, obs, reward_sum, last_done, cost_sum, last_result, auto_reset, max_episode_steps,
                               0, h->n);
    p.n_steps = n_steps; p.random_policy = actions ? 0 : 1; p.act_stride = h->n; p.policy_seed = policy_seed;
    p.done_count = done_count; p.actions_out = actions_out;
    p.trunc = nullptr; p.final_obs = nullptr;              // per-step episode ends have no place in a rollout's sums
    if (attach_record(h, p, n_steps, "ngw_rollout")) return 1;   // (the per-step ones go to the record)
    CK(cudaSetDevice(h->device));
    before_device_call(h, (cudaStream_t)stream);
    return launch_step(h, p, (cudaStream_t)stream);
}

int ngw_rollout_policy(ngw_handle* h, const int32_t* weights, const int32_t* bias, int32_t n_policy_actions,
                       int32_t n_steps, void* obs, float* reward_sum, float* cost_sum, int32_t* done_count,
                       uint8_t* last_done, uint8_t* last_result, int32_t* actions_out, int32_t auto_reset,
                       int32_t max_episode_steps, void* stream) {
    if (!h) return fail("null handle");
    if (!weights || !bias || n_policy_actions < 1 || n_policy_actions > 16)
        return fail("ngw_rollout_policy: need weights, bias and 1..16 policy actions");
    if (h->obs_dim == 0 || !obs) return fail("ngw_rollout_policy: needs a LidarInFront observation (and an obs buffer)");
    if (h->obs_format != NGW_OBS_I32)
        return fail("ngw_rollout_policy: the linear policy reads int32 observation rows (NGW_OBS_I32)");
    if (n_steps < 1) return fail("ngw_rollout_policy: n_steps must be >= 1");
    if (!reward_sum || !cost_sum || !last_done || !last_result) return fail("ngw_rollout_policy: null output pointer");
    if ((uintptr_t)obs & 15) return fail("ngw_rollout_policy: obs must be 16-byte aligned");
    StepParams p = step_params(h, reinterpret_cast<const int32_t*>(h->zero_byte), obs, reward_sum, last_done, cost_sum,
                               last_result, auto_reset, max_episode_steps, 0, h->n);
    p.n_steps = n_steps; p.random_policy = 0; p.act_stride = h->n; p.done_count = done_count; p.actions_out = actions_out;
    p.policy_w = weights; p.policy_b = bias; p.policy_actions = n_policy_actions;
    p.trunc = nullptr; p.final_obs = nullptr;
    if (attach_record(h, p, n_steps, "ngw_rollout_policy")) return 1;
    CK(cudaSetDevice(h->device));
    before_device_call(h, (cudaStream_t)stream);
    return launch_step(h, p, (cudaStream_t)stream);
}

int ngw_observe(ngw_handle* h, void* obs, void* stream) {
    if (!h) return fail("null handle");
    if (h->obs_dim == 0) return 0;
    if (!obs || ((uintptr_t)obs & 15)) return fail("ngw_observe: obs must be a 16-byte aligned device pointer");
    CK(cudaSetDevice(h->device));
    before_device_call(h, (cudaStream_t)stream);
    return launch_step(h, step_params(h, nullptr, obs, nullptr, nullptr, nullptr, nullptr, 0, 0, 0, h->n),
                       (cudaStream_t)stream);
}

// Device staging of the host-buffer path: ONE block  observation rows [n] | pad to 16 | reward | step_cost | done | result
// (n-element sections), so that a caller whose host buffers have the same layout gets a whole step with ONE device-to-host
// copy (ngw_host_layout gives the offsets).
static size_t host_small_offset(const ngw_handle* h) { return ((size_t)h->n * h->obs_row_bytes + 15) & ~(size_t)15; }

static int ensure_host_path(ngw_handle* h) {
    if (!h->hs) {
        CK(cudaStreamCreateWithFlags(&h->hs, cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&h->ev_dev, cudaEventDisableTiming));
        CK(cudaMalloc(&h->h_actions, (size_t)h->np * 4));
    }
    const size_t off = host_small_offset(h), need = off + (size_t)h->n * 10 + 64;
    if (need != h->h_obs_bytes) {                                   // (re)built for the current observation format
        CK(cudaStreamSynchronize(h->hs));
        cudaFree(h->h_obs);
        h->h_obs = nullptr; h->h_obs_bytes = 0;
        CK(cudaMalloc(&h->h_obs, need));
        h->h_obs_bytes = need;
        unsigned char* small = h->h_obs + off;
        h->h_reward = reinterpret_cast<float*>(small);
        h->h_cost = reinterpret_cast<float*>(small + (size_t)h->n * 4);
        h->h_done = small + (size_t)h->n * 8;
        h->h_result = small + (size_t)h->n * 9;
    }
    return 0;
}

int ngw_set_message_buffer(ngw_handle* h, uint16_t* msg_dev) {
    if (!h) return fail("null handle");
    h->msg = msg_dev;
    return 0;
}

int ngw_set_episode_end_buffers(ngw_handle* h, uint8_t* truncated_dev, void* final_obs_dev) {
    if (!h) return fail("null handle");
    if ((uintptr_t)final_obs_dev & 15) return fail("ngw_set_episode_end_buffers: final_obs must be 16-byte aligned");
    h->trunc = truncated_dev;
    h->final_obs = static_cast<unsigned char*>(final_obs_dev);
    return 0;
}

int ngw_set_rollout_record(ngw_handle* h, const ngw_rollout_record* rec) {
    if (!h) return fail("null handle");
    if (!rec) { h->rec_on = false; h->rec = ngw_rollout_record{}; return 0; }
    if (rec->max_steps < 1) return fail("ngw_set_rollout_record: max_steps must be >= 1");
    if (h->obs_dim > 0 && (((uintptr_t)rec->obs & 15) || ((uintptr_t)rec->final_obs & 15)))
        return fail("ngw_set_rollout_record: obs and final_obs must be 16-byte aligned");
    if (((uintptr_t)rec->reward & 3) || ((uintptr_t)rec->step_cost & 3))
        return fail("ngw_set_rollout_record: reward and step_cost must be 4-byte aligned");
    h->rec = *rec;
    h->rec_on = true;
    return 0;
}

int ngw_step_host_end(ngw_handle* h) {
    if (!h) return fail("null handle");
    if (!h->hs) return 0;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->hs));
    h->host_dirty = false;
    return 0;
}

int ngw_step_host(ngw_handle* h, const int32_t* actions, void* obs, float* reward, uint8_t* done, float* step_cost,
                  uint8_t* result, int32_t auto_reset, int32_t max_episode_steps) {
    if (ngw_step_host_begin(h, actions, obs, reward, done, step_cost, result, auto_reset, max_episode_steps)) return 1;
    return ngw_step_host_end(h);
}

int ngw_step_host_begin(ngw_handle* h, const int32_t* actions, void* obs, float* reward, uint8_t* done,
                        float* step_cost, uint8_t* result, int32_t auto_reset, int32_t max_episode_steps) {
    if (!h) return fail("null handle");
    if (!actions || !reward || !done || !step_cost || !result) return fail("ngw_step_host: null pointer");
    CK(cudaSetDevice(h->device));
    if (ensure_host_path(h)) return 1;
    cudaStream_t s = h->hs;
    if (h->dev_dirty) {
        // a reset / load_state / device-path step was enqueued on the caller's stream since the last host-path call:
        // this step must see its result (ngw_reset followed by ngw_step_host is the reference-facing pattern)
        cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
        if (cudaStreamIsCapturing(h->last_dev_stream, &cap) != cudaSuccess) { cudaGetLastError(); cap = cudaStreamCaptureStatusNone; }
        if (cap == cudaStreamCaptureStatusNone) {
            if (cudaEventRecord(h->ev_dev, h->last_dev_stream) == cudaSuccess) CK(cudaStreamWaitEvent(s, h->ev_dev, 0));
            else { cudaGetLastError(); CK(cudaDeviceSynchronize()); }
        }
        h->dev_dirty = false;
    }
    // The step kernel is a small fraction of the PCIe time of its own outputs, so chunked compute/copy overlap buys
    // nothing: one stream, one H2D, one launch, two D2H; overlap comes from pipelining several handles (_begin/_end).
    long long n = h->n;
    size_t cnt = (size_t)n;
    CK(cudaMemcpyAsync(h->h_actions, actions, cnt * 4, cudaMemcpyHostToDevice, s));
    if (launch_step(h, step_params(h, h->h_actions, h->h_obs, h->h_reward, h->h_done, h->h_cost, h->h_result,
                                   auto_reset, max_episode_steps, 0, n), s)) return 1;
    h->host_dirty = true;
    const unsigned char* r8 = reinterpret_cast<const unsigned char*>(reward);
    const bool small_packed = reinterpret_cast<const unsigned char*>(step_cost) == r8 + cnt * 4 && done == r8 + cnt * 8 &&
                              result == r8 + cnt * 9;
    if (h->obs_dim > 0 && obs && small_packed && r8 == static_cast<const unsigned char*>(obs) + host_small_offset(h)) {
        // the caller's buffers mirror the staging block: the whole step leaves with one copy
        CK(cudaMemcpyAsync(obs, h->h_obs, host_small_offset(h) + cnt * 10, cudaMemcpyDeviceToHost, s));
        return 0;
    }
    if (h->obs_dim > 0 && obs)
        CK(cudaMemcpyAsync(obs, h->h_obs, cnt * h->obs_row_bytes, cudaMemcpyDeviceToHost, s));
    if (small_packed) {
        CK(cudaMemcpyAsync(reward, h->h_reward, cnt * 10, cudaMemcpyDeviceToHost, s));   // same layout: one copy
    } else {
        CK(cudaMemcpyAsync(reward, h->h_reward, cnt * 4, cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(done, h->h_done, cnt, cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(step_cost, h->h_cost, cnt * 4, cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(result, h->h_result, cnt, cudaMemcpyDeviceToHost, s));
    }
    return 0;
}

int ngw_agent_map(ngw_handle* h, int8_t* out, int32_t view, void* stream) {
    if (!h || !out || view < 1 || view > 32) return fail("ngw_agent_map: bad arguments");
    CK(cudaSetDevice(h->device));
    before_device_call(h, (cudaStream_t)stream);
    long long total = h->n * (2 * view + 1) * (2 * view + 1);
    agent_map_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(h->map, h->pose, out, h->n, h->ms,
                                                                                         view);
    h->launches++;
    CK(cudaGetLastError());
    return 0;
}

int ngw_stats(ngw_handle* h, double* out8_dev, int32_t reset_after, void* stream) {
    if (!h || !out8_dev) return fail("ngw_stats: null");
    CK(cudaSetDevice(h->device));
    before_device_call(h, (cudaStream_t)stream);
    stats_fold_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(h->stats, out8_dev, reset_after);
    h->launches++;
    CK(cudaGetLastError());
    return 0;
}

int64_t ngw_launch_count(ngw_handle* h) { return h ? h->launches : 0; }
int64_t ngw_concurrent_launch_count(ngw_handle* h) { return h ? h->concurrent_launches : 0; }

}  // extern "C"
