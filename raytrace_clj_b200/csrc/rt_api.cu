// rt_api.cu — host side of libraytrace_b200.so: the C ABI of include/raytrace_b200.h.
//
// One rt_ctx owns, per CUDA device: the scene in "cull order" SoA buffers, a float sum buffer,
// an 8-bit image buffer, counters and a stream.  There is no CPU rendering path anywhere in
// this file: every entry point that produces results launches sm_100a kernels.
#include "../../include/raytrace_b200.h"

#include <cuda_runtime.h>
#include <dlfcn.h>
#include <math_constants.h>
#include <nccl.h>   // types only: the library itself is dlopen'ed when a multi-device context asks for the NCCL reduce

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <mutex>
#include <thread>
#include <string>
#include <vector>

#include "rt_bvh_build.cuh"
#include "rt_kernels.cuh"
#include "rt_scene_build.cuh"

using namespace rt;

namespace {

constexpr int kR = 4;          // rays (path slots) per thread
constexpr int kBlock = 256;
constexpr int kMinBlocks = 1;     // megakernel: NO register cap — capped at 128 registers it spilled 288 bytes and one path in ~600 k
                                  // differed from run to run (the uncapped build is bit-reproducible and agrees with the wavefront)
constexpr int kTileCap = 4096; // float4 slots of the shared-memory sphere tile when the scene is tiled

thread_local std::string g_create_error;

struct DeviceBuffers {
    int dev = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_done = nullptr;
    // scene (the device blob and its pinned staging copy are reused across rt_set_scene calls)
    void* scene_blob = nullptr;
    void* scene_stage = nullptr;
    size_t scene_bytes = 0;
    size_t scene_used = 0;                // bytes of the current scene's blob
    // rt_set_scene_device: the listed leaves' FP64 bounding spheres stay on the device (c0, c1, r; t0t1 and flags are the
    // blob's), in the layout the device BVH build reads
    void* bs_buf = nullptr;
    size_t bs_bytes = 0;
    BvhLeafInput bs_in{};
    void* sb_scratch = nullptr;           // device 0: radii, sort storage, candidates, cull order of the device build
    size_t sb_scratch_bytes = 0;
    SbResult* h_sb = nullptr;             // pinned: the validation / direct-sphere result read back before the blob is laid out
    cudaEvent_t ev_sb = nullptr;          // orders the build after the caller's stream
    DevScene sc{};
    // frame
    float* d_sum = nullptr;
    float* d_mean = nullptr;
    uint8_t* d_rgb8 = nullptr;
    size_t frame_px = 0;
    unsigned long long* d_counters = nullptr;   // DC_COUNT + 1 (last = work counter)
    // wavefront queues
    struct WaveLane {
        float4* queue = nullptr;            // 2 * 3 * entries float4
        unsigned long long* best = nullptr; // 2 * entries
        uint2* pairs = nullptr;
        uint2* cands = nullptr;
        double* cand_t = nullptr;
        unsigned* cand_count = nullptr;
        WaveState* state = nullptr;
        LaneStatus* h_status = nullptr;     // pinned + mapped: written by the device (publish_status), polled by the host
        LaneStatus* d_status = nullptr;     // its device address
        cudaEvent_t ev_done = nullptr;
        cudaStream_t stream = nullptr;      // lane 0 runs on the caller's stream, the others on their own
        cudaStream_t stage_stream = nullptr;   // high priority: refine / tie-break / shade of this lane (RT_CULL_CLAIMS > 0)
        cudaEvent_t ev_culled = nullptr, ev_shaded = nullptr;
        size_t entries = 0;
        bool best_clean = false;            // every closest-hit word is (+inf, MISS): true after a render ran to completion
    } lanes[kMaxLanes];
    cudaEvent_t ev_lane_start = nullptr;
    // timeline trace (RT_TRACE): one record per wavefront kernel launch of the last render
    TraceRec* d_trace = nullptr;
    struct TraceMeta { const char* kernel; int lane, iter; };
    std::vector<TraceMeta> trace_meta;
    // scratch for diagnostics
    void* scratch = nullptr;
    size_t scratch_bytes = 0;
    int sm_count = 0, clock_khz = 0;
    char name[64] = {0};
    float last_ms = 0.f;
    bool timed = false;
    // RT_ACCEL_BVH: the flattened tree (4 float4 per node), rebuilt with the scene / the movers' time window
    float4* bvh_nodes = nullptr;
    size_t bvh_cap = 0;
    int bvh_builder = 0, bvh_depth = 0;   // the published tree: 0 host / 1 device builder, depth of its deepest leaf
    long long bvh_build_ns = 0;           // device build: CUDA-event time of the last one (upload included)
    void* bvh_scratch = nullptr;          // device build: inputs, leaf boxes, codes, parents, flags, sort storage (grown on demand)
    size_t bvh_scratch_bytes = 0;
    int* h_bvh_depth = nullptr;           // pinned: the built tree's depth, read back before the tree is published
    cudaEvent_t ev_b0 = nullptr, ev_b1 = nullptr;
    // pinned staging for the results of rt_render (root device): D2H at link speed, then one host memcpy into the caller's buffer
    void* h_stage = nullptr;
    size_t h_stage_bytes = 0;
    cudaEvent_t ev_r0 = nullptr, ev_r1 = nullptr;   // around the cross-device reduce (RT_CTR_REDUCE_NS)
    cudaEvent_t ev_chunk[4] = {};                   // D2H of the results in chunks: the host memcpy of chunk k overlaps the copy of chunk k + 1
};

// NCCL, loaded on demand (single process, one communicator per device: ncclCommInitAll)
struct NcclApi {
    void* handle = nullptr;
    ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*Reduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    std::vector<ncclComm_t> comms;
};

}  // namespace

// Tuning knobs of one context.  The RT_* environment variables give the defaults at rt_create; rt_set_option changes
// them per context afterwards (two contexts of one process can differ).
struct Options {
    int wave_lanes = 2;               // RT_WAVE_LANES: independent halves of the path population (1..kMaxLanes)
    long long wave_capacity = 1ll << 24;   // RT_WAVE_CAPACITY: paths in flight per device, all lanes together
    int cull_claims = 2;              // RT_CULL_CLAIMS: batches a cull warp takes before it retires (0 = persistent warps)
    int cull_ctas_per_sm = 4;         // RT_CULL_CTAS_PER_SM
    int cull_shape = 0;               // RT_CULL_SHAPE: 0 = 128x5 (default), 1 = 128x6, 2 = 256x2
    int light_block = 128;            // RT_LIGHT_BLOCK: CTA size of the stage kernels
    long long tail_entries = 1 << 19; // RT_TAIL_ENTRIES: queue length at which wf_tail takes over
    int tail_ctas_per_sm = 0;         // RT_TAIL_CTAS_PER_SM (0 = automatic)
    int tile_records = 1024;          // RT_TILE_RECORDS
    int direct_spheres = 1;           // RT_DIRECT_SPHERES
    int common_origin = 1;            // RT_COMMON_ORIGIN
    int reduce = 0;                   // multi-device rt_render: 0 = NVLink peer loads inside the resolve kernel, 1 = ncclReduce
    int rows = 0;                     // multi-device partition: 0 = sample slices, 1 = interleaved rows
    int tail_block = 256;             // RT_TAIL_BLOCK: CTA size of the tail kernel (32 | 64 | 128 | 256)
    int tail_rays = 1;                // RT_TAIL_RAYS: rays per thread of the tail kernel's cull while its slices are long (1 | 4)
    int tail_solo = 24;               // RT_TAIL_SOLO: a tail slice of this many paths or fewer is finished one lane group per path (0 = staged to the end)
    int tail_lpp = 32;                // RT_TAIL_LPP: lanes of such a group (8 | 16 | 32)
    int mega_regcap = 0;              // 1: the register-capped megakernel (128 registers, 2 CTAs / SM) instead of the uncapped one
    int wave_depth = 2;               // RT_WAVE_DEPTH: iterations the host keeps queued ahead of the GPU per lane
    int cull_tc = 1;                  // RT_CULL_TC: 0 = FP32 cull (wf_cull) always; 1 = the cull runs on the tensor cores (wf_cull_tc) when the list fits (<= 1024 leaves);
                                      //   2 = except a lane's first, all-camera-ray iteration when those rays share an origin
    int tc_tiles_per_cta = 0;         // RT_TC_TILES_PER_CTA: ray tiles a wf_cull_tc CTA takes before it retires (0 = one CTA per SM, persistent)
    int tc_ctas = 0;                  // RT_TC_CTAS: persistent wf_cull_tc CTAs (0 = one per SM); fewer leaves whole SMs to the other lane's stage kernels
    int bvh_build = 1;                // RT_BVH_BUILD: RT_ACCEL_BVH's tree built on the host (0), on the device (2), or on the device
                                      //   from kBvhDeviceMinLeaves listed leaves up (1)
};

struct rt_ctx {
    std::mutex mu;
    std::string err;
    std::vector<DeviceBuffers> devs;
    Options opt;
    bool has_scene = false, has_cam = false;
    int n_spheres = 0;            // world primitives
    int n_total = 0;              // + boundary primitives of media
    int n_list = 0, n_cull = 0;   // spheres in the cull list / cull records (padded)
    int cull_cap = 0, preloaded = 0;
    int tc_tiles = 0;             // feature tiles (256 leaves each) of the tensor-core cull; over 4, an iteration takes several launches
    std::vector<std::vector<float>> tc_scratch_rows;   // build_cull_records: the leaves' feature rows before they are placed
    std::vector<int> tc_row_k;    // feature row -> cull index (-1 = padding): a fixed shuffle, so every 64-row block sees the same mix
    int generic = 0;              // some leaf is not a plain sphere (rt_set_scene_ex)
    int accel = RT_ACCEL_BRUTE_FORCE;
    bool bvh_dirty = true;        // the tree must be (re)built before the next BVH render
    // time window [win_lo, win_hi] the movers' bounding spheres cover; grown (and the cull records rebuilt)
    // when a camera shutter interval or a traced ray's time falls outside
    double win_lo = 0.0, win_hi = 0.0;
    std::vector<float> h_c0r, h_c1, h_t0t1;   // geometry in cull order (world primitives, then boundary primitives)
    std::vector<unsigned> h_flags;
    // world-space bounding sphere of every world leaf, cull order: centre at t0 / t1 (equal unless moving), radius
    std::vector<double> h_bs_c0, h_bs_c1, h_bs_r;
    // rt_set_scene_device: the bounding spheres live on every device (DeviceBuffers::bs_in); h_bs_*, h_t0t1 and h_flags are
    // a mirror downloaded on demand (bs_mirror), and tc_row_k / tc_scratch_rows are unused (the rows are in the blob)
    bool bs_on_device = false, bs_mirror = false;
    bool any_moving = false;      // some listed or direct sphere moves (rt_set_scene_device)
    DevCamera cam{};
    std::atomic<uint64_t> n_launches{0};
    std::mutex err_mu;
    bool profile = false;
    double stage_ms[4] = {0, 0, 0, 0};   // cull, refine, tie-break, shade (profile mode)
    double reduce_ms = 0.0;              // cross-device reduce of the multi-device renders since the last reset
    std::vector<bool> peer_ok;
    NcclApi nccl;
};

namespace {

int fail(rt_ctx* ctx, int code, const std::string& msg) {
    if (ctx) {
        std::lock_guard<std::mutex> lk(ctx->err_mu);   // device worker threads may fail concurrently
        ctx->err = msg;
    } else {
        g_create_error = msg;
    }
    return code;
}

#define RT_CUDA(ctx, expr)                                                                          \
    do {                                                                                            \
        cudaError_t e__ = (expr);                                                                   \
        if (e__ != cudaSuccess)                                                                     \
            return fail(ctx, RT_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e__));     \
    } while (0)

int ensure_scratch(rt_ctx* ctx, DeviceBuffers& d, size_t bytes) {
    if (d.scratch_bytes >= bytes) return RT_OK;
    if (d.scratch) cudaFree(d.scratch);
    d.scratch = nullptr;
    d.scratch_bytes = 0;
    RT_CUDA(ctx, cudaMalloc(&d.scratch, bytes));
    d.scratch_bytes = bytes;
    return RT_OK;
}

int ensure_frame(rt_ctx* ctx, DeviceBuffers& d, size_t px) {
    if (d.frame_px >= px) return RT_OK;
    if (d.d_sum) cudaFree(d.d_sum);
    if (d.d_mean) cudaFree(d.d_mean);
    if (d.d_rgb8) cudaFree(d.d_rgb8);
    d.d_sum = d.d_mean = nullptr;
    d.d_rgb8 = nullptr;
    d.frame_px = 0;
    RT_CUDA(ctx, cudaMalloc(&d.d_sum, px * 3 * sizeof(float)));
    RT_CUDA(ctx, cudaMalloc(&d.d_mean, px * 3 * sizeof(float)));
    RT_CUDA(ctx, cudaMalloc(&d.d_rgb8, px * 3));
    d.frame_px = px;
    return RT_OK;
}


void free_lane(DeviceBuffers::WaveLane& L) {
    if (L.queue) cudaFree(L.queue);
    if (L.best) cudaFree(L.best);
    if (L.pairs) cudaFree(L.pairs);
    if (L.cands) cudaFree(L.cands);
    if (L.cand_t) cudaFree(L.cand_t);
    if (L.cand_count) cudaFree(L.cand_count);
    L.queue = nullptr; L.best = nullptr; L.pairs = nullptr; L.cands = nullptr; L.cand_t = nullptr; L.cand_count = nullptr;
    L.entries = 0;
}

void free_wave(DeviceBuffers& d) {
    for (auto& L : d.lanes) {
        free_lane(L);
        if (L.state) cudaFree(L.state);
        if (L.h_status) cudaFreeHost(L.h_status);
        if (L.ev_done) cudaEventDestroy(L.ev_done);
        if (L.stream) cudaStreamDestroy(L.stream);
        if (L.stage_stream) cudaStreamDestroy(L.stage_stream);
        if (L.ev_culled) cudaEventDestroy(L.ev_culled);
        if (L.ev_shaded) cudaEventDestroy(L.ev_shaded);
        L = DeviceBuffers::WaveLane();
    }
    if (d.ev_lane_start) cudaEventDestroy(d.ev_lane_start);
    d.ev_lane_start = nullptr;
    if (d.d_trace) cudaFree(d.d_trace);
    d.d_trace = nullptr;
}

int ensure_lane(rt_ctx* ctx, DeviceBuffers& d, int lane, size_t entries) {
    DeviceBuffers::WaveLane& L = d.lanes[lane];
    if (!L.state) {
        RT_CUDA(ctx, cudaMalloc(&L.state, sizeof(WaveState)));
        RT_CUDA(ctx, cudaHostAlloc(&L.h_status, sizeof(LaneStatus), cudaHostAllocMapped));
        RT_CUDA(ctx, cudaHostGetDevicePointer((void**)&L.d_status, L.h_status, 0));
        RT_CUDA(ctx, cudaEventCreateWithFlags(&L.ev_done, cudaEventDisableTiming));
        if (lane > 0) RT_CUDA(ctx, cudaStreamCreateWithFlags(&L.stream, cudaStreamNonBlocking));
        int prio_least = 0, prio_greatest = 0;
        RT_CUDA(ctx, cudaDeviceGetStreamPriorityRange(&prio_least, &prio_greatest));
        RT_CUDA(ctx, cudaStreamCreateWithPriority(&L.stage_stream, cudaStreamNonBlocking, prio_greatest));
        RT_CUDA(ctx, cudaEventCreateWithFlags(&L.ev_culled, cudaEventDisableTiming));
        RT_CUDA(ctx, cudaEventCreateWithFlags(&L.ev_shaded, cudaEventDisableTiming));
        if (!d.ev_lane_start) RT_CUDA(ctx, cudaEventCreateWithFlags(&d.ev_lane_start, cudaEventDisableTiming));
    }
    if (L.entries >= entries) return RT_OK;
    free_lane(L);
    RT_CUDA(ctx, cudaMalloc(&L.queue, entries * 2 * 3 * sizeof(float4)));
    RT_CUDA(ctx, cudaMalloc(&L.best, entries * 2 * sizeof(unsigned long long)));
    RT_CUDA(ctx, cudaMalloc(&L.pairs, entries * kPairsPerEntry * sizeof(uint2)));
    // candidate regions are private to the warps of the refine grid: pair_cap rounded up per warp
    const size_t cand_slots = entries * kPairsPerEntry + (size_t)d.sm_count * 8 * 8 * 32;
    RT_CUDA(ctx, cudaMalloc(&L.cands, cand_slots * sizeof(uint2)));
    RT_CUDA(ctx, cudaMalloc(&L.cand_t, cand_slots * sizeof(double)));
    RT_CUDA(ctx, cudaMalloc(&L.cand_count, (size_t)d.sm_count * 8 * 8 * sizeof(unsigned)));
    L.entries = entries;
    L.best_clean = false;
    return RT_OK;
}

size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

float round_up_f32(double x) {
    float f = (float)x;
    if ((double)f < x) f = nextafterf(f, INFINITY);
    return f;
}

size_t mega_smem_bytes(int cull_cap) { return (size_t)cull_cap * sizeof(float4) + Culler<kR, kBlock>::LIST_BYTES; }

template <typename Kern>
int configure_kernel(rt_ctx* ctx, Kern kern, size_t smem, int* blocks_per_sm) {
    RT_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int b = 0;
    RT_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, kern, kBlock, smem));
    if (b < 1) return fail(ctx, RT_ERR_CUDA, "kernel does not fit on an SM");
    *blocks_per_sm = b;
    return RT_OK;
}

long long env_ll(const char* name, long long dflt) {
    const char* v = getenv(name);
    return (v && *v) ? atoll(v) : dflt;
}
int env_int(const char* name, int dflt) { return (int)env_ll(name, dflt); }

Options options_from_env() {
    Options o;
    o.wave_lanes = env_int("RT_WAVE_LANES", o.wave_lanes);
    o.wave_capacity = env_ll("RT_WAVE_CAPACITY", o.wave_capacity);
    o.cull_claims = env_int("RT_CULL_CLAIMS", o.cull_claims);
    o.cull_ctas_per_sm = env_int("RT_CULL_CTAS_PER_SM", o.cull_ctas_per_sm);
    const char* shape = getenv("RT_CULL_SHAPE");
    if (shape && !strcmp(shape, "128x6")) o.cull_shape = 1;
    if (shape && !strcmp(shape, "256x2")) o.cull_shape = 2;
    o.light_block = env_int("RT_LIGHT_BLOCK", o.light_block);
    o.tail_entries = env_ll("RT_TAIL_ENTRIES", o.tail_entries);
    o.tail_ctas_per_sm = env_int("RT_TAIL_CTAS_PER_SM", o.tail_ctas_per_sm);
    o.tile_records = env_int("RT_TILE_RECORDS", o.tile_records);
    o.direct_spheres = env_int("RT_DIRECT_SPHERES", o.direct_spheres);
    o.common_origin = env_int("RT_COMMON_ORIGIN", o.common_origin);
    o.reduce = env_int("RT_REDUCE", o.reduce);
    o.rows = env_int("RT_ROWS", o.rows);
    o.wave_depth = env_int("RT_WAVE_DEPTH", o.wave_depth);
    o.tail_rays = env_int("RT_TAIL_RAYS", o.tail_rays);
    o.tail_solo = env_int("RT_TAIL_SOLO", o.tail_solo);
    o.tail_lpp = env_int("RT_TAIL_LPP", o.tail_lpp);
    o.tail_block = env_int("RT_TAIL_BLOCK", o.tail_block);
    o.cull_tc = env_int("RT_CULL_TC", o.cull_tc);
    o.tc_tiles_per_cta = env_int("RT_TC_TILES_PER_CTA", o.tc_tiles_per_cta);
    o.tc_ctas = env_int("RT_TC_CTAS", o.tc_ctas);
    o.bvh_build = env_int("RT_BVH_BUILD", o.bvh_build);
    return o;
}

// Wavefront render of one device's share: enqueue iterations (cull, refine, shade) ahead of the
// GPU and poll the queue count every kWaveChunk iterations; returns when the queue has drained (the last
// polled chunk may still be finishing its empty kernels).
template <int BLOCK, int MINB>
int cull_config(rt_ctx* ctx, size_t* smem, int* bps, void (**kern)(const WaveParams)) {
    *kern = wf_cull<kR, BLOCK, MINB>;
    // a resident scene keeps two tiles (general + common-origin records); a tiled scene streams ONE tile and the loader
    // writes whichever form the batch needs
    *smem = (ctx->preloaded ? 2 : 1) * (size_t)ctx->cull_cap * sizeof(float4) + Culler<kR, BLOCK>::LIST_BYTES;
    RT_CUDA(ctx, cudaFuncSetAttribute(*kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)*smem));
    RT_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(bps, *kern, BLOCK, *smem));
    if (*bps < 1) return fail(ctx, RT_ERR_CUDA, "cull kernel does not fit on an SM");
    return RT_OK;
}

// Wavefront render of one device's share.  The path population is split into `lanes` independent halves,
// each running its own cull -> refine -> tie-break -> shade sequence on its own stream over its own queues
// (they share only the work counter and the frame, both atomics): one lane's FP32-issue-bound cull kernel
// co-runs with the other lane's latency-bound refine / shade kernels.  The host enqueues kWaveChunk
// iterations per lane ahead of the GPU and polls each lane's queue count; when the work counter is
// exhausted and a lane's queue is short, one wf_tail launch finishes that lane (every CTA on its own slice).
int launch_wave(rt_ctx* ctx, DeviceBuffers& d, const RenderParams& P, unsigned long long, cudaStream_t stream) {
    // CTA shape of the cull kernel (threads x register-cap CTAs/SM): 128x5 (default) | 128x6 | 256x2
    const Options& opt = ctx->opt;
    void (*cull)(const WaveParams) = nullptr;
    size_t smem = 0;
    int bps = 0, cull_block = 256, rc;
    if (opt.cull_shape == 2) rc = cull_config<256, 2>(ctx, &smem, &bps, &cull);
    else if (opt.cull_shape == 1) { rc = cull_config<128, 6>(ctx, &smem, &bps, &cull); cull_block = 128; }
    else { rc = cull_config<128, 5>(ctx, &smem, &bps, &cull); cull_block = 128; }
    if (rc) return rc;
    const int cull_ctas_env = opt.cull_ctas_per_sm;                       // one fewer than the occupancy limit leaves
    if (cull_ctas_env > 0) bps = std::min(bps, cull_ctas_env);           // room for the other lane's light kernels
    const size_t cap_env = (size_t)std::max<long long>(64, opt.wave_capacity);
    const int lanes_env = std::max(1, std::min(kMaxLanes, opt.wave_lanes));
    const int n_lanes = (ctx->profile || P.total_work < 65536) ? 1 : lanes_env;   // stage timing wants one lane
    const size_t capacity = align_up((size_t)std::min<unsigned long long>(cap_env / n_lanes, (P.total_work + n_lanes - 1) / n_lanes), 32);

    // tail kernel: one CTA per SM per lane (two lanes' tails run side by side)
    bool done[kMaxLanes] = {};
    const unsigned tail_entries = (unsigned)std::max<long long>(0, opt.tail_entries);
    const bool gen = ctx->generic != 0;   // GEN = false instantiations hold none of the generic-leaf / extended-texture code
    const bool tail4 = opt.tail_rays == 4;
    // CTA size of the tail kernel: every CTA finishes its own slice, __syncthreads() between the stages.  Smaller CTAs =
    // more, shorter slices and cheaper barriers (32: one warp per CTA, the barrier is warp-local and the stages of
    // different warps overlap on the SM)
    const int tail_block = (gen || tail4) ? 256 : (opt.tail_block == 32 || opt.tail_block == 64 || opt.tail_block == 128 ? opt.tail_block : 256);
    const size_t tail_smem = (size_t)ctx->cull_cap * sizeof(float4) +
                             (tail4 ? Culler<4, 256>::LIST_BYTES : (size_t)Culler<1, 256>::LIST_WORDS * tail_block * sizeof(uint32_t));
    int tail_bps = 0;
    void (*k_tail)(const WaveParams) = gen ? wf_tail<256, true, 1> : (tail4 ? wf_tail<256, false, 4> : wf_tail<256, false, 1>);
    if (tail_block == 128) k_tail = wf_tail<128, false, 1>;
    if (tail_block == 64) k_tail = wf_tail<64, false, 1>;
    if (tail_block == 32) k_tail = wf_tail<32, false, 1>;
    void (*k_refine)(const WaveParams) = gen ? wf_refine<true> : wf_refine<false>;
    void (*k_shade)(const WaveParams) = gen ? wf_shade<true> : wf_shade<false>;
    RT_CUDA(ctx, cudaFuncSetAttribute(k_tail, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tail_smem));
    RT_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&tail_bps, k_tail, tail_block, tail_smem));
    // automatic: the same number of tail THREADS per SM whatever the CTA size (256 per lane with two lanes, 512 with one)
    const int tail_auto = (n_lanes > 1 ? 1 : std::max(1, std::min((int)(tail_bps * tail_block / 256), 2))) * (256 / tail_block);
    const int tail_grid = d.sm_count * (opt.tail_ctas_per_sm > 0 ? opt.tail_ctas_per_sm : tail_auto);
    const bool bvh = ctx->accel == RT_ACCEL_BVH;   // closest hit through the tree: one wf_bvh launch instead of cull + refine + tie-break
    void (*k_bvh)(const WaveParams) = gen ? wf_bvh<true> : wf_bvh<false>;
    const bool tail_ok = tail_bps >= 1 && tail_entries > 0 && !ctx->profile && !bvh;
    // tensor-core cull (rt_cull_tc.cuh): one 544-thread CTA per SM, the whole sphere-feature list resident in shared memory
    // (below ~160 leaves most of a 256-column feature tile is padding and the FP32 loop wins: C5-100 39.7 vs 48.0 ms, Cornell box
    // 47.8 vs 64.0 ms; cull_tc = 3 forces the tensor-core kernel whatever the list length)
    // Scenes with generic leaves (rectangles, boxes, triangles, media: rt_set_scene_ex) stay on the FP32 loop too: their bounding
    // spheres are loose, a ray's line meets dozens of them, the per-warp candidate lists overflow and the overflow path (exact
    // re-intersection of the ray in wf_shade) takes over: make-final 1.47 s on the FP32 loop, 2.96 s on the tensor cores.
    const bool use_tc = opt.cull_tc != 0 && ctx->tc_tiles > 0 && !bvh && ((ctx->n_list >= tc::MIN_LEAVES && !ctx->generic) || opt.cull_tc == 3);
    const int tc_launch_tiles = std::min(ctx->tc_tiles, (int)tc::MAX_TILES);
    const int tc_slots = tc::slots_for(tc_launch_tiles, 227 * 1024);
    const size_t tc_smem = tc::smem_bytes(tc_launch_tiles, tc_slots);
    if (use_tc) RT_CUDA(ctx, cudaFuncSetAttribute(wf_cull_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc_smem));
    const int tc_per_cta = std::max(0, opt.tc_tiles_per_cta);
    const int tc_grid = opt.tc_ctas > 0 ? std::min(opt.tc_ctas, 4 * d.sm_count) : d.sm_count;
    // one launch per 1024 leaves of the list ("pass"): the pairs of all passes pile up in the same buffer
    auto launch_tc = [&](const WaveParams& Wl, int per_cta, unsigned ctas, cudaStream_t s_) {
        WaveParams Wt = Wl;
        Wt.claims_per_warp = per_cta;
        Wt.tc_slots = tc_slots;
        for (int t0 = 0, pass = 0; t0 < ctx->tc_tiles; t0 += tc::MAX_TILES, ++pass) {
            Wt.tc_tile0 = t0;
            Wt.tc_launch_tiles = std::min((int)tc::MAX_TILES, ctx->tc_tiles - t0);
            Wt.tc_pass = pass;
            wf_cull_tc<<<ctas, tc::THREADS, tc_smem, s_>>>(Wt);
            if (pass) ctx->n_launches += 1;
        }
    };

    const int light_block = std::max(64, std::min(256, opt.light_block / 32 * 32));   // <= a cull CTA in every resource
    const int light_grid = d.sm_count * 8 * 256 / light_block;
    const int cull_grid = d.sm_count * bps;
    // RT_CULL_CLAIMS = k > 0 (resident scenes): cull warps retire after k batches — the cull becomes many short CTAs, SM
    // slots turn over every few tens of microseconds, and the OTHER lane's refine / tie-break / shade kernels, launched
    // on a high-priority stream, take the freed slots at once instead of waiting for the whole persistent cull to end.
    // 0 = persistent cull warps, one stream per lane.
    const int claims_env = std::max(0, opt.cull_claims);
    const int claims = (ctx->profile || !ctx->preloaded || n_lanes < 2 || bvh) ? 0 : claims_env;
    const int cull_warps = cull_block / 32, resident_warps = cull_grid * cull_warps;
    unsigned n_bound[kMaxLanes];   // upper bound of each lane's queue length (sizes the short-CTA grids)
    WaveParams W[kMaxLanes];
    cudaStream_t st[kMaxLanes];
    unsigned long long first = 0;
    for (int l = 0; l < n_lanes; ++l) {
        if ((rc = ensure_lane(ctx, d, l, capacity))) return rc;
        DeviceBuffers::WaveLane& L = d.lanes[l];
        W[l] = WaveParams{};
        W[l].base = P;
        W[l].queue[0] = L.queue;
        W[l].queue[1] = L.queue + 3 * capacity;
        W[l].best_t = L.best;
        W[l].best_key = L.best + L.entries;   // fixed split: the words stay reset from one render to the next
        W[l].pairs = L.pairs;
        W[l].cands = L.cands;
        W[l].cand_t = L.cand_t;
        W[l].cand_count = L.cand_count;
        W[l].st = L.state;
        W[l].capacity = (int)capacity;
        W[l].pair_cap = (unsigned)std::min<size_t>(capacity * kPairsPerEntry, 0xfffffff0u);
        W[l].cur = 0;
        W[l].claims_per_warp = claims;
        W[l].resident_warps = claims ? resident_warps : 0;
        W[l].tail_solo = (unsigned)std::max(0, opt.tail_solo);
        W[l].tail_lpp = opt.tail_lpp == 8 ? 8u : (opt.tail_lpp == 16 ? 16u : 32u);
        st[l] = l == 0 ? stream : L.stream;
    }
    // RT_TRACE=<file>: device-side timeline of this render's kernels (dumped by the next rt_get_counters)
    static const char* trace_path = getenv("RT_TRACE");
    constexpr int kTraceMax = 8192;
    const bool tracing = trace_path && *trace_path;
    if (tracing) {
        if (!d.d_trace) RT_CUDA(ctx, cudaMalloc(&d.d_trace, kTraceMax * sizeof(TraceRec)));
        static const std::vector<TraceRec> init((size_t)kTraceMax, TraceRec{~0ull, 0ull});
        RT_CUDA(ctx, cudaMemcpyAsync(d.d_trace, init.data(), init.size() * sizeof(TraceRec), cudaMemcpyHostToDevice, stream));
        d.trace_meta.clear();
    }
    auto trace_slot = [&](const char* kernel, int lane, int iter) -> TraceRec* {
        if (!tracing || (int)d.trace_meta.size() >= kTraceMax) return nullptr;
        d.trace_meta.push_back({kernel, lane, iter});
        return d.d_trace + (d.trace_meta.size() - 1);
    };
    int iter_no[kMaxLanes] = {};
    // RT_DEBUG_SYNC=1: synchronise after every launch of the iteration loop and name the kernel that failed
    static const bool debug_sync = getenv("RT_DEBUG_SYNC") && *getenv("RT_DEBUG_SYNC") == '1';
    auto dbg = [&](const char* what, int lane, int it) -> int {
        if (!debug_sync) return RT_OK;
        cudaError_t e = cudaDeviceSynchronize();
        if (e != cudaSuccess) return fail(ctx, RT_ERR_CUDA, std::string(what) + " (lane " + std::to_string(lane) + ", iteration " + std::to_string(it) + "): " + cudaGetErrorString(e));
        return RT_OK;
    };
    // the shared work counter starts past every lane's first fill
    unsigned count0[kMaxLanes];
    unsigned long long total0 = 0;
    for (int l = 0; l < n_lanes; ++l) {
        count0[l] = (unsigned)std::min<unsigned long long>(capacity, P.total_work - total0);
        total0 += count0[l];
        n_bound[l] = count0[l];
    }
    InitParams I{};
    I.n_lanes = n_lanes;
    I.work_counter = P.work_counter;
    I.counters = P.counters;
    I.total0 = total0;
    I.total_work = P.total_work;
    for (int l = 0; l < n_lanes; ++l) {
        DeviceBuffers::WaveLane& L = d.lanes[l];
        I.st[l] = L.state;
        I.first[l] = first;
        I.count[l] = count0[l];
        first += count0[l];
        if (!L.best_clean) {   // after an allocation / an aborted render; wf_shade keeps the words reset otherwise
            wf_fill_best<<<d.sm_count * 4, 256, 0, stream>>>(L.best, L.best + L.entries, L.entries);
            ctx->n_launches += 1;
        }
        L.best_clean = false;   // until this render has run to completion
    }
    wf_init<<<1, 1, 0, stream>>>(I);
    ctx->n_launches += 1;
    RT_CUDA(ctx, cudaGetLastError());
    RT_CUDA(ctx, cudaEventRecord(d.ev_lane_start, stream));
    for (int l = 1; l < n_lanes; ++l) RT_CUDA(ctx, cudaStreamWaitEvent(st[l], d.ev_lane_start, 0));

    // The host only keeps the GPU fed: it queues `depth` iterations ahead per lane (cull, refine, tie-break, shade) and
    // watches each lane's status record, which the device writes straight into mapped host memory (publish_status: no
    // copy, no event, nothing in the lane's stream).  How much fresh work an iteration gets and when a lane is finished are
    // decided on the device; kernels queued past the end return at once.  When the status says that no new work can appear
    // and the queue is short, ONE wf_tail launch (behind the iterations already queued) finishes the lane.
    const int depth = std::max(1, std::min(16, opt.wave_depth));
    int enq[kMaxLanes] = {}, seen[kMaxLanes] = {};
    bool tailed[kMaxLanes] = {};
    for (int l = 0; l < n_lanes; ++l) {
        DeviceBuffers::WaveLane& L = d.lanes[l];
        memset(L.h_status, 0, sizeof(LaneStatus));
        W[l].status = L.d_status;
        if (count0[l] == 0) done[l] = true;
    }
    std::vector<cudaEvent_t> evs;   // profile mode (one lane): 5 events per iteration
    unsigned idle_spins = 0;
    for (;;) {
        bool progressed = false, all_done = true;
        for (int l = 0; l < n_lanes; ++l) {
            if (done[l]) continue;
            all_done = false;
            DeviceBuffers::WaveLane& L = d.lanes[l];
            while (!tailed[l] && enq[l] - seen[l] < depth) {
                cudaEvent_t e[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
                if (ctx->profile)
                    for (auto& x : e) { RT_CUDA(ctx, cudaEventCreate(&x)); evs.push_back(x); }
                if (ctx->profile) cudaEventRecord(e[0], st[l]);
                W[l].iter = (unsigned)(enq[l] + 1);
                // cull_tc = 2: a lane's first iteration (only fresh camera rays) stays on the FP32 cull's common-origin form when they
                // share an origin.  Faster for that launch alone (1.18 vs 1.4 ms for 9.6 M rays), slower for the frame (5.93 vs 5.72 ms
                // on C2: the short-CTA FP32 cull and the other lane's tensor-core cull get in each other's way)
                const bool tc_now = use_tc && !(enq[l] == 0 && P.common_origin && opt.cull_tc == 2);
                if (bvh) {
                    W[l].trace = trace_slot("bvh", l, iter_no[l]);
                    k_bvh<<<light_grid, 128, 0, st[l]>>>(W[l]);
                    if (ctx->profile) { cudaEventRecord(e[1], st[l]); cudaEventRecord(e[2], st[l]); cudaEventRecord(e[3], st[l]); }
                    W[l].trace = trace_slot("shade", l, iter_no[l]);
                    k_shade<<<light_grid, light_block, 0, st[l]>>>(W[l]);
                    if (ctx->profile) cudaEventRecord(e[4], st[l]);
                    ctx->n_launches -= 2;   // two launches this iteration, not four
                } else if (claims) {
                    W[l].trace = trace_slot("cull", l, iter_no[l]);
                    if (debug_sync) {
                        WaveState hs{};
                        cudaMemcpy(&hs, W[l].st, sizeof hs, cudaMemcpyDeviceToHost);
                        fprintf(stderr, "lane %d iteration %d cur %d: in flight %u fresh %u | other queue %u %u | mode %u exhausted %u npairs %u\n", l, enq[l], W[l].cur,
                                hs.cnt[W[l].cur][0], hs.cnt[W[l].cur][1], hs.cnt[W[l].cur ^ 1][0], hs.cnt[W[l].cur ^ 1][1], hs.mode, hs.exhausted, hs.npairs);
                    }
                    if (tc_now) {
                        const unsigned tiles = (n_bound[l] + tc::TILE_M - 1) / tc::TILE_M;
                        const unsigned ctas = tc_per_cta ? (tiles + (unsigned)tc_per_cta - 1u) / (unsigned)tc_per_cta : (unsigned)tc_grid;
                        launch_tc(W[l], tc_per_cta, std::max(1u, ctas), st[l]);
                    } else {
                    // every work item of the launch must find a warp: items <= n / (32 R) + 2 resident_warps + 8 (wf_cull_body)
                    const unsigned items = n_bound[l] / (32u * kR) + 2u * (unsigned)resident_warps + 8u;
                    const unsigned ctas = (items + (unsigned)(cull_warps * claims) - 1u) / (unsigned)(cull_warps * claims);
                    cull<<<ctas, cull_block, smem, st[l]>>>(W[l]);
                    }
                    if ((rc = dbg(tc_now ? "wf_cull_tc" : "wf_cull", l, enq[l]))) return rc;
                    RT_CUDA(ctx, cudaEventRecord(L.ev_culled, st[l]));
                    RT_CUDA(ctx, cudaStreamWaitEvent(L.stage_stream, L.ev_culled, 0));
                    W[l].trace = trace_slot("refine", l, iter_no[l]);
                    k_refine<<<light_grid, light_block, 0, L.stage_stream>>>(W[l]);
                    if ((rc = dbg("wf_refine", l, enq[l]))) return rc;
                    W[l].trace = trace_slot("tiebreak", l, iter_no[l]);
                    wf_tiebreak<<<light_grid, light_block, 0, L.stage_stream>>>(W[l]);
                    if ((rc = dbg("wf_tiebreak", l, enq[l]))) return rc;
                    W[l].trace = trace_slot("shade", l, iter_no[l]);
                    k_shade<<<light_grid, light_block, 0, L.stage_stream>>>(W[l]);
                    if ((rc = dbg("wf_shade", l, enq[l]))) return rc;
                    RT_CUDA(ctx, cudaEventRecord(L.ev_shaded, L.stage_stream));
                    RT_CUDA(ctx, cudaStreamWaitEvent(st[l], L.ev_shaded, 0));
                } else {
                    W[l].trace = trace_slot("cull", l, iter_no[l]);
                    if (tc_now) {
                        launch_tc(W[l], 0, (unsigned)tc_grid, st[l]);
                    } else {
                        cull<<<cull_grid, cull_block, smem, st[l]>>>(W[l]);
                    }
                    if (ctx->profile) cudaEventRecord(e[1], st[l]);
                    W[l].trace = trace_slot("refine", l, iter_no[l]);
                    k_refine<<<light_grid, light_block, 0, st[l]>>>(W[l]);
                    if (ctx->profile) cudaEventRecord(e[2], st[l]);
                    W[l].trace = trace_slot("tiebreak", l, iter_no[l]);
                    wf_tiebreak<<<light_grid, light_block, 0, st[l]>>>(W[l]);
                    if (ctx->profile) cudaEventRecord(e[3], st[l]);
                    W[l].trace = trace_slot("shade", l, iter_no[l]);
                    k_shade<<<light_grid, light_block, 0, st[l]>>>(W[l]);
                    if (ctx->profile) cudaEventRecord(e[4], st[l]);
                }
                RT_CUDA(ctx, cudaGetLastError());
                W[l].cur ^= 1;
                ++iter_no[l];
                ctx->n_launches += 4;
                ++enq[l];
                progressed = true;
            }
        }
        if (all_done) break;
        for (int l = 0; l < n_lanes; ++l) {
            if (done[l]) continue;
            DeviceBuffers::WaveLane& L = d.lanes[l];
            const volatile LaneStatus* hs = L.h_status;
            const unsigned seq = hs->seq;
            if ((int)seq == seen[l] && hs->mode != MODE_DONE) continue;
            std::atomic_thread_fence(std::memory_order_acquire);
            const unsigned n_next = hs->n_next, n_fresh = hs->n_fresh, exhausted = hs->exhausted, mode = hs->mode;
            if (hs->seq != seq) continue;   // the device was writing the next record: read it on the next round
            seen[l] = (int)seq;
            progressed = true;
            if (exhausted) n_bound[l] = std::min(n_bound[l], n_next);   // from here on a lane's population only shrinks
            if (mode == MODE_DONE) { done[l] = true; continue; }
            if (tail_ok && !tailed[l] && exhausted && n_fresh == 0 && n_next <= tail_entries) {
                // no new work can appear and the queue is short: one launch, behind the iterations already queued
                // (they shrink the population further; the tail takes whatever is left), finishes this lane
                W[l].iter = (unsigned)(enq[l] + 1);
                W[l].trace = trace_slot("tail", l, iter_no[l]);
                k_tail<<<tail_grid, tail_block, tail_smem, st[l]>>>(W[l]);
                if ((rc = dbg("wf_tail", l, enq[l]))) return rc;
                RT_CUDA(ctx, cudaGetLastError());
                ctx->n_launches += 1;
                tailed[l] = true;
            }
        }
        if (!progressed) {   // nothing to queue, nothing new: spin briefly, then yield the core
            if (++idle_spins > 200) {
                if (cudaSuccess != cudaPeekAtLastError()) RT_CUDA(ctx, cudaGetLastError());
                if (idle_spins > 20000 && (idle_spins % 1000) == 0) {   // a lost lane would spin forever: ask the stream
                    for (int l = 0; l < n_lanes; ++l)
                        if (!done[l] && cudaStreamQuery(st[l]) == cudaSuccess && d.lanes[l].h_status->seq == (unsigned)seen[l] &&
                            enq[l] > seen[l])
                            return fail(ctx, RT_ERR_CUDA, "wavefront lane finished its queue without reporting status");
                }
                std::this_thread::yield();
            }
        } else {
            idle_spins = 0;
        }
    }
    // the caller's stream continues only after every lane has drained
    for (int l = 1; l < n_lanes; ++l) {
        RT_CUDA(ctx, cudaEventRecord(d.lanes[l].ev_done, st[l]));
        RT_CUDA(ctx, cudaStreamWaitEvent(stream, d.lanes[l].ev_done, 0));
    }
    for (int l = 0; l < n_lanes; ++l) d.lanes[l].best_clean = true;   // every entry was consumed (and its words reset) by wf_shade / wf_tail
    if (ctx->profile) {
        RT_CUDA(ctx, cudaStreamSynchronize(stream));
        for (size_t i = 0; i + 4 < evs.size(); i += 5)
            for (int sgi = 0; sgi < 4; ++sgi) {
                float ms = 0.f;
                if (cudaEventElapsedTime(&ms, evs[i + sgi], evs[i + sgi + 1]) == cudaSuccess) ctx->stage_ms[sgi] += ms;
            }
        for (auto x : evs) cudaEventDestroy(x);
    }
    return RT_OK;
}

int launch_params(rt_ctx* ctx, DeviceBuffers& d, RenderParams& P, int variant, cudaStream_t stream);

// Launch the render kernels for one device's share of the work (async on d.stream).
int launch_render(rt_ctx* ctx, DeviceBuffers& d, int nx, int ny, int sample_begin, int sample_count, int row_offset,
                  int row_stride, int max_depth, uint64_t seed, int variant, float* d_sum, cudaStream_t stream) {
    RenderParams P{};
    P.sc = d.sc;
    P.cam = ctx->cam;
    P.nx = nx;
    P.ny = ny;
    P.sample_begin = sample_begin;
    P.sample_count = sample_count;
    P.row_offset = row_offset;
    P.row_stride = row_stride;
    P.rows_in_shard = (ny - row_offset + row_stride - 1) / row_stride;
    P.max_depth = max_depth;
    P.key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
    P.sum = d_sum;
    P.counters = d.d_counters;
    P.work_counter = d.d_counters + DC_COUNT;
    P.total_work = (unsigned long long)sample_count * (unsigned long long)nx * (unsigned long long)P.rows_in_shard;
    if ((sample_begin + sample_count) >= (1 << 24)) return fail(ctx, RT_ERR_ARG, "sample index must stay below 2^24");
    return launch_params(ctx, d, P, variant, stream);
}

// P: scene-independent fields filled by the caller (frame, work, seed, outputs); the rest is completed here
int launch_params(rt_ctx* ctx, DeviceBuffers& d, RenderParams& P, int variant, cudaStream_t stream) {
    if (variant != RT_VARIANT_MEGAKERNEL && variant != RT_VARIANT_WAVEFRONT)
        return fail(ctx, RT_ERR_ARG, "unknown render variant");
    if (variant == RT_VARIANT_WAVEFRONT && P.max_depth > 255)
        return fail(ctx, RT_ERR_ARG, "the wavefront variant packs the depth in 8 bits: max_depth <= 255");
    P.sc = d.sc;
    P.cam = ctx->cam;
    P.counters = d.d_counters;
    P.work_counter = d.d_counters + DC_COUNT;
    P.cull_cap = ctx->cull_cap;
    P.preloaded = ctx->preloaded;
    P.common_origin = (ctx->opt.common_origin && (ctx->cam.type == CAM_PINHOLE || ctx->cam.lens_radius == 0.f)) ? 1 : 0;
    RT_CUDA(ctx, cudaMemsetAsync(P.work_counter, 0, sizeof(unsigned long long), stream));
    if (P.total_work == 0) return RT_OK;
    size_t smem = mega_smem_bytes(ctx->cull_cap);
    unsigned long long want = (P.total_work + (unsigned long long)kBlock * kR - 1) / ((unsigned long long)kBlock * kR);
    int bps = 0;
    if (variant == RT_VARIANT_MEGAKERNEL) {
        // option "mega_regcap" = 1: the 128-register build of round 1 (2 CTAs / SM, spills) kept as an A/B for the
        // reproducibility check (tests/test_gpu_parity.py::test_render_is_reproducible runs both)
        void (*kern)(const RenderParams) = ctx->generic ? mega_kernel<kR, kBlock, kMinBlocks, true>
                                           : (ctx->opt.mega_regcap ? mega_kernel<kR, kBlock, 2, false> : mega_kernel<kR, kBlock, kMinBlocks, false>);
        int rc = configure_kernel(ctx, kern, smem, &bps);
        if (rc) return rc;
        int grid = (int)std::min<unsigned long long>((unsigned long long)d.sm_count * bps, want);
        if (grid < 1) grid = 1;
        kern<<<grid, kBlock, smem, stream>>>(P);
        RT_CUDA(ctx, cudaGetLastError());
        ctx->n_launches += 1;
        return RT_OK;
    }
    // persistent wavefront: every CTA is an independent engine with its own queues
    return launch_wave(ctx, d, P, want, stream);
}

// FP32 cull record per listed sphere: (-cx, -cy, -cz, W = r^2 inflated - c.c) (Culler, rt_kernels.cuh).  A moving
// sphere (hitable.clj:224-259) is represented by the bounding sphere of its swept volume over [win_lo, win_hi]:
// centre = midpoint of centre(win_lo), centre(win_hi), radius = r + half the travelled distance.  The inflation
// covers the float rounding of the record itself and the sphere's share of the cull's rounding budget
// (48 u c.c + 8 u r^2, u = 2^-24; the bound is 32.6 u c.c + 4.1 u r^2), so the cull only ever over-reports.
// Records [n_list, n_cull) are padding: W = -inf, the key is -inf for every ray.  The direct spheres' records
// follow the padding (used as a pre-test where those spheres are resolved).
// tc_out (or null): the tensor-core cull's TF32 feature rows of the listed leaves (rt_cull_tc.cuh: sphere_slots), tc_tiles
// tiles of 256 rows in the canonical UMMA layout — same bounding spheres, with that kernel's own rounding budget in W
// (96 u c.c + 24 u R2 on top of the geometric inflation).
void build_cull_records(rt_ctx* ctx, double win_lo, double win_hi, float* cull_all, float* tc_out) {
    const double eps = std::ldexp(1.0, -20), u = std::ldexp(1.0, -24);
    for (int i = 0; i < ctx->n_spheres; ++i) {
        // listed spheres at [0, n_list); the direct spheres' records follow the padding, at n_cull + (i - n_list)
        float* cull_a = i < ctx->n_list ? cull_all : cull_all + 4 * (size_t)(ctx->n_cull - ctx->n_list);
        // the leaf's world-space bounding sphere (a sphere: itself; a rectangle / triangle / medium: the sphere around it,
        // carried through the leaf's wrappers at upload)
        double r = std::fabs(ctx->h_bs_r[(size_t)i]);
        double mid[3], half2 = 0.0, cmax = 0.0;
        const bool moving = (ctx->h_flags[i] & RT_SPHERE_MOVING) != 0;
        for (int c = 0; c < 3; ++c) {
            double p0 = ctx->h_bs_c0[3 * (size_t)i + c];
            if (moving) {
                double p1 = ctx->h_bs_c1[3 * (size_t)i + c], t0 = ctx->h_t0t1[2 * i], t1 = ctx->h_t0t1[2 * i + 1];
                double fa = (win_lo - t0) / (t1 - t0), fb = (win_hi - t0) / (t1 - t0);
                double pa = p0 * (1.0 - fa) + p1 * fa, pb = p0 * (1.0 - fb) + p1 * fb;
                mid[c] = 0.5 * (pa + pb);
                half2 += 0.25 * (pb - pa) * (pb - pa);
            } else {
                mid[c] = p0;
            }
            cmax = std::max(cmax, std::fabs(mid[c]));
        }
        double rb = r + std::sqrt(half2);
        // float rounding of the midpoint (+ margin); generic leaves: also the rounding of the transformed centre / radius
        double e = (moving || ctx->generic) ? std::ldexp(1.0, -21) * (cmax + rb) : 0.0;
        double cc = 0.0;
        for (int c = 0; c < 3; ++c) {
            const float neg = (float)(-mid[c]);       // negated: the chains are seeded FFMAs on -c
            cull_a[4 * i + c] = neg;
            cc += (double)neg * (double)neg;          // c.c of the record AS STORED
        }
        double re = rb + e;
        double r2i = re * re * (1.0 + eps) + 48.0 * u * cc + 8.0 * u * re * re;
        cull_a[4 * i + 3] = round_up_f32(r2i - cc);
        if (tc_out && i < ctx->n_list) {
            const double c[3] = {-(double)cull_a[4 * i], -(double)cull_a[4 * i + 1], -(double)cull_a[4 * i + 2]};   // the centre AS STORED
            const double Wtc = re * re * (1.0 + eps) + 96.0 * u * cc + 24.0 * u * re * re - cc;
            float row[tc::KTOT];
            tc::sphere_slots(c, Wtc, row);
            ctx->tc_scratch_rows[(size_t)i].assign(row, row + tc::KTOT);
        }
    }
    for (int k = ctx->n_list; k < ctx->n_cull; ++k) {
        cull_all[4 * k] = cull_all[4 * k + 1] = cull_all[4 * k + 2] = 0.f;
        cull_all[4 * k + 3] = -INFINITY;
    }
    if (tc_out) {
        float pad[tc::KTOT];
        tc::padding_slots(pad);
        for (int p = 0; p < ctx->tc_tiles * tc::TILE_N; ++p) {
            const int k = ctx->tc_row_k[(size_t)p];
            const float* row = k >= 0 ? ctx->tc_scratch_rows[(size_t)k].data() : pad;
            float* tile = tc_out + (size_t)(p / tc::TILE_N) * (tc::B_TILE_BYTES / 4);
            for (int q = 0; q < tc::KTOT; ++q) tile[tc::canon_off(tc::TILE_N, p % tc::TILE_N, q) / 4] = row[q];
        }
    }
}

// build_cull_records on one device over its device-resident bounding spheres (a scene of rt_set_scene_device): the FP32
// records, the padding records and the tensor-core feature rows of the rows the blob's tc_row_k deals out
int enqueue_records_device(rt_ctx* ctx, DeviceBuffers& d, double win_lo, double win_hi) {
    const int n = ctx->n_spheres, pad = ctx->n_cull - ctx->n_list, rows = ctx->tc_tiles * tc::TILE_N;
    sb_cull_records<<<(n + pad + kSbBlock - 1) / kSbBlock, kSbBlock, 0, d.stream>>>(d.bs_in, n, ctx->n_list, ctx->n_cull, win_lo, win_hi,
                                                                                    const_cast<float4*>(d.sc.cull_a));
    if (rows)
        sb_tc_rows<<<(rows + kSbBlock - 1) / kSbBlock, kSbBlock, 0, d.stream>>>(d.bs_in, d.sc.tc_row_k, rows, win_lo, win_hi,
                                                                                const_cast<float*>(d.sc.cull_tc));
    RT_CUDA(ctx, cudaGetLastError());
    return RT_OK;
}

// make sure the movers' bounding spheres cover ray times in [lo, hi]
int ensure_window(rt_ctx* ctx, double lo, double hi) {
    if (lo >= ctx->win_lo && hi <= ctx->win_hi) return RT_OK;
    if (!(lo <= hi) || !std::isfinite(lo) || !std::isfinite(hi)) return fail(ctx, RT_ERR_ARG, "ray time is not finite");
    ctx->win_lo = std::min(ctx->win_lo, lo);
    ctx->win_hi = std::max(ctx->win_hi, hi);
    if (ctx->bs_on_device) {   // rt_set_scene_device: the records are rebuilt where the bounding spheres are
        if (!ctx->any_moving) return RT_OK;
        ctx->bvh_dirty = true;
        for (auto& d : ctx->devs) {
            RT_CUDA(ctx, cudaSetDevice(d.dev));
            RT_CUDA(ctx, cudaDeviceSynchronize());   // a render enqueued with sync = 0 on a caller's stream may still read the records
            if (int rc = enqueue_records_device(ctx, d, ctx->win_lo, ctx->win_hi)) return rc;
        }
        for (auto& d : ctx->devs) {
            RT_CUDA(ctx, cudaSetDevice(d.dev));
            RT_CUDA(ctx, cudaStreamSynchronize(d.stream));
        }
        cudaSetDevice(ctx->devs[0].dev);
        return RT_OK;
    }
    bool any_moving = false;
    for (unsigned f : ctx->h_flags) any_moving |= (f & RT_SPHERE_MOVING) != 0;
    if (!any_moving) return RT_OK;
    ctx->bvh_dirty = true;   // the movers' boxes cover the window too
    std::vector<float> cull((size_t)(ctx->n_cull + ctx->n_spheres - ctx->n_list) * 4);
    std::vector<float> tcr((size_t)ctx->tc_tiles * (tc::B_TILE_BYTES / 4));
    build_cull_records(ctx, ctx->win_lo, ctx->win_hi, cull.data(), tcr.empty() ? nullptr : tcr.data());
    if (cull.empty()) return RT_OK;
    for (auto& d : ctx->devs) {
        RT_CUDA(ctx, cudaSetDevice(d.dev));
        RT_CUDA(ctx, cudaDeviceSynchronize());   // a render enqueued with sync = 0 on a caller's stream may still read the records
        RT_CUDA(ctx, cudaMemcpy((void*)d.sc.cull_a, cull.data(), cull.size() * sizeof(float), cudaMemcpyHostToDevice));
        if (!tcr.empty()) RT_CUDA(ctx, cudaMemcpy((void*)d.sc.cull_tc, tcr.data(), tcr.size() * sizeof(float), cudaMemcpyHostToDevice));
    }
    cudaSetDevice(ctx->devs[0].dev);
    return RT_OK;
}

// RT_ACCEL_BVH: build the tree over the listed leaves on the host — the reference's make-bvh shape (hitable.clj:108-123:
// sort along one axis, the left half takes ceil(n/2), a lone leaf is stored as both children) with the axis chosen as
// the longest extent of the centroids instead of at random — and upload it.  Leaf boxes = the boxes of the leaves' world-
// space bounding spheres over the movers' time window, widened so the FP32 slab test can only over-report.
struct BuildLeaf {
    float lo[3], hi[3];
    float c[3];
    int k;
};
int bvh_build_node(std::vector<BuildLeaf>& L, int begin, int end, std::vector<float>& nodes, float lo[3], float hi[3], int depth,
                   int* max_depth) {
    if (end - begin == 1) {
        for (int a = 0; a < 3; ++a) { lo[a] = L[(size_t)begin].lo[a]; hi[a] = L[(size_t)begin].hi[a]; }
        *max_depth = std::max(*max_depth, depth);
        return ~L[(size_t)begin].k;
    }
    float cmin[3] = {INFINITY, INFINITY, INFINITY}, cmax[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int i = begin; i < end; ++i)
        for (int a = 0; a < 3; ++a) { cmin[a] = std::min(cmin[a], L[(size_t)i].c[a]); cmax[a] = std::max(cmax[a], L[(size_t)i].c[a]); }
    int axis = 0;
    for (int a = 1; a < 3; ++a) if (cmax[a] - cmin[a] > cmax[axis] - cmin[axis]) axis = a;
    const int mid = begin + (end - begin + 1) / 2;
    std::nth_element(L.begin() + begin, L.begin() + mid, L.begin() + end,
                     [axis](const BuildLeaf& x, const BuildLeaf& y) { return x.c[axis] < y.c[axis]; });
    const size_t me = nodes.size() / 16;
    nodes.resize(nodes.size() + 16, 0.f);
    float llo[3], lhi[3], rlo[3], rhi[3];
    const int left = bvh_build_node(L, begin, mid, nodes, llo, lhi, depth + 1, max_depth);
    const int right = bvh_build_node(L, mid, end, nodes, rlo, rhi, depth + 1, max_depth);
    float* N = nodes.data() + 16 * me;
    N[0] = llo[0]; N[1] = llo[1]; N[2] = llo[2]; N[3] = lhi[0]; N[4] = lhi[1]; N[5] = lhi[2];
    N[6] = rlo[0]; N[7] = rlo[1]; N[8] = rlo[2]; N[9] = rhi[0]; N[10] = rhi[1]; N[11] = rhi[2];
    memcpy(&N[12], &left, 4);
    memcpy(&N[13], &right, 4);
    for (int a = 0; a < 3; ++a) { lo[a] = std::min(llo[a], rlo[a]); hi[a] = std::max(lhi[a], rhi[a]); }
    return (int)me;
}

int ensure_bvh_nodes(rt_ctx* ctx, DeviceBuffers& d, size_t bytes) {
    if (d.bvh_cap >= bytes) return RT_OK;
    if (d.bvh_nodes) cudaFree(d.bvh_nodes);
    d.bvh_nodes = nullptr;
    d.bvh_cap = 0;
    RT_CUDA(ctx, cudaMalloc(&d.bvh_nodes, bytes));
    d.bvh_cap = bytes;
    return RT_OK;
}

// a scene of rt_set_scene_device keeps its bounding spheres on the device; the host builder reads a mirror, downloaded
// from the first device once per scene
int ensure_bs_mirror(rt_ctx* ctx) {
    if (!ctx->bs_on_device || ctx->bs_mirror) return RT_OK;
    const DeviceBuffers& d = ctx->devs[0];
    const size_t n = (size_t)ctx->n_spheres;
    ctx->h_bs_c0.resize(3 * n);
    ctx->h_bs_c1.resize(3 * n);
    ctx->h_bs_r.resize(n);
    ctx->h_t0t1.resize(2 * n);
    ctx->h_flags.resize(n);
    RT_CUDA(ctx, cudaSetDevice(d.dev));
    RT_CUDA(ctx, cudaMemcpy(ctx->h_bs_c0.data(), d.bs_in.c0, 3 * n * 8, cudaMemcpyDeviceToHost));
    RT_CUDA(ctx, cudaMemcpy(ctx->h_bs_c1.data(), d.bs_in.c1, 3 * n * 8, cudaMemcpyDeviceToHost));
    RT_CUDA(ctx, cudaMemcpy(ctx->h_bs_r.data(), d.bs_in.r, n * 8, cudaMemcpyDeviceToHost));
    RT_CUDA(ctx, cudaMemcpy(ctx->h_t0t1.data(), d.bs_in.t0t1, 2 * n * 4, cudaMemcpyDeviceToHost));
    RT_CUDA(ctx, cudaMemcpy(ctx->h_flags.data(), d.bs_in.flags, n * 4, cudaMemcpyDeviceToHost));
    ctx->bs_mirror = true;
    return RT_OK;
}

int bvh_build_host(rt_ctx* ctx) {
    if (int rc = ensure_bs_mirror(ctx)) return rc;
    const int n = ctx->n_list;
    std::vector<BuildLeaf> L((size_t)n);
    for (int k = 0; k < n; ++k) {
        BuildLeaf& b = L[(size_t)k];
        b.k = k;
        const bool moving = (ctx->h_flags[(size_t)k] & RT_SPHERE_MOVING) != 0;
        const double r = std::fabs(ctx->h_bs_r[(size_t)k]);
        for (int a = 0; a < 3; ++a) {
            double pa = ctx->h_bs_c0[3 * (size_t)k + a], pb = pa;
            if (moving) {
                const double p0 = ctx->h_bs_c0[3 * (size_t)k + a], p1 = ctx->h_bs_c1[3 * (size_t)k + a];
                const double t0 = ctx->h_t0t1[2 * k], t1 = ctx->h_t0t1[2 * k + 1];
                const double fa = (ctx->win_lo - t0) / (t1 - t0), fb = (ctx->win_hi - t0) / (t1 - t0);
                pa = p0 * (1.0 - fa) + p1 * fa;
                pb = p0 * (1.0 - fb) + p1 * fb;
            }
            const double lo = std::min(pa, pb) - r, hi = std::max(pa, pb) + r;
            const double m = 1e-6 * (std::fabs(lo) + std::fabs(hi) + r) + 1e-30;   // covers the float rounding of the box and its share of the slab test
            b.lo[a] = nextafterf((float)(lo - m), -INFINITY);
            b.hi[a] = nextafterf((float)(hi + m), INFINITY);
            b.c[a] = (float)(0.5 * (lo + hi));
        }
    }
    std::vector<float> nodes;
    nodes.reserve(16 * (size_t)std::max(1, n));
    float lo[3], hi[3];
    int depth = 1;
    if (n == 1) {   // a lone leaf is both children of the root (hitable.clj:113-114)
        nodes.assign(16, 0.f);
        for (int a = 0; a < 3; ++a) { nodes[(size_t)a] = nodes[6 + (size_t)a] = L[0].lo[a]; nodes[3 + (size_t)a] = nodes[9 + (size_t)a] = L[0].hi[a]; }
        const int leaf = ~0;
        memcpy(&nodes[12], &leaf, 4);
        memcpy(&nodes[13], &leaf, 4);
    } else {
        const int root = bvh_build_node(L, 0, n, nodes, lo, hi, 0, &depth);
        if (root != 0) return fail(ctx, RT_ERR_STATE, "BVH build: the root is not node 0");
    }
    for (auto& d : ctx->devs) {
        RT_CUDA(ctx, cudaSetDevice(d.dev));
        RT_CUDA(ctx, cudaDeviceSynchronize());
        const size_t bytes = nodes.size() * sizeof(float);
        if (int rc = ensure_bvh_nodes(ctx, d, bytes)) return rc;
        RT_CUDA(ctx, cudaMemcpy(d.bvh_nodes, nodes.data(), bytes, cudaMemcpyHostToDevice));
        d.sc.bvh = d.bvh_nodes;
        d.sc.bvh_nodes = (int)(nodes.size() / 16);
        d.bvh_builder = 0;
        d.bvh_depth = depth;
        d.bvh_build_ns = 0;
    }
    cudaSetDevice(ctx->devs[0].dev);
    return RT_OK;
}

// RT_ACCEL_BVH on the device (rt_bvh_build.cuh): enqueue the whole build on one device's stream, the depth read back into
// pinned memory last.  The tree lands in the node buffer; it is published (or replaced by the host build, when too deep)
// after the stream has finished.
int bvh_enqueue_device(rt_ctx* ctx, DeviceBuffers& d) {
    const int n = ctx->n_list;
    const int n_nodes = std::max(1, n - 1);
    RT_CUDA(ctx, cudaSetDevice(d.dev));
    RT_CUDA(ctx, cudaDeviceSynchronize());   // a render enqueued with sync = 0 on a caller's stream may still read the tree
    if (int rc = ensure_bvh_nodes(ctx, d, (size_t)n_nodes * 4 * sizeof(float4))) return rc;
    size_t sort_bytes = 0;
    RT_CUDA(ctx, cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, (const unsigned long long*)nullptr, (unsigned long long*)nullptr,
                                                 (const int*)nullptr, (int*)nullptr, n, 0, 3 * (int)kMortonAxisBits, d.stream));
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off = align_up(off + bytes, 256); return o; };
    const size_t n_ = (size_t)n;
    const size_t o_c0 = take(n_ * 3 * 8), o_c1 = take(n_ * 3 * 8), o_r = take(n_ * 8), o_t = take(n_ * 2 * 4), o_fl = take(n_ * 4);
    const size_t o_box = take(n_ * 6 * 4), o_cb = take(6 * 4), o_code = take(n_ * 8), o_code2 = take(n_ * 8);
    const size_t o_leaf = take(n_ * 4), o_leaf2 = take(n_ * 4), o_par = take((2 * n_ - 1) * 4), o_arr = take((size_t)n_nodes * 4);
    const size_t o_h = take((size_t)n_nodes * 4), o_depth = take(4), o_sort = take(sort_bytes);
    if (d.bvh_scratch_bytes < off) {
        if (d.bvh_scratch) cudaFree(d.bvh_scratch);
        d.bvh_scratch = nullptr;
        d.bvh_scratch_bytes = 0;
        RT_CUDA(ctx, cudaMalloc(&d.bvh_scratch, off));
        d.bvh_scratch_bytes = off;
    }
    if (!d.h_bvh_depth) {
        RT_CUDA(ctx, cudaHostAlloc(&d.h_bvh_depth, sizeof(int), cudaHostAllocDefault));
        RT_CUDA(ctx, cudaEventCreate(&d.ev_b0));
        RT_CUDA(ctx, cudaEventCreate(&d.ev_b1));
    }
    char* S = (char*)d.bvh_scratch;
    const cudaStream_t st = d.stream;
    // a scene of rt_set_scene_device: the bounding spheres are already on this device
    const BvhLeafInput in = ctx->bs_on_device ? d.bs_in
                                              : BvhLeafInput{(const double*)(S + o_c0), (const double*)(S + o_c1), (const double*)(S + o_r),
                                                             (const float*)(S + o_t), (const unsigned*)(S + o_fl)};
    float* boxes = (float*)(S + o_box);
    unsigned* cb = (unsigned*)(S + o_cb);
    int* depth = (int*)(S + o_depth);
    RT_CUDA(ctx, cudaEventRecord(d.ev_b0, st));
    if (!ctx->bs_on_device) {
        RT_CUDA(ctx, cudaMemcpyAsync(S + o_c0, ctx->h_bs_c0.data(), n_ * 3 * 8, cudaMemcpyHostToDevice, st));
        RT_CUDA(ctx, cudaMemcpyAsync(S + o_c1, ctx->h_bs_c1.data(), n_ * 3 * 8, cudaMemcpyHostToDevice, st));
        RT_CUDA(ctx, cudaMemcpyAsync(S + o_r, ctx->h_bs_r.data(), n_ * 8, cudaMemcpyHostToDevice, st));
        RT_CUDA(ctx, cudaMemcpyAsync(S + o_t, ctx->h_t0t1.data(), n_ * 2 * 4, cudaMemcpyHostToDevice, st));
        RT_CUDA(ctx, cudaMemcpyAsync(S + o_fl, ctx->h_flags.data(), n_ * 4, cudaMemcpyHostToDevice, st));
    }
    RT_CUDA(ctx, cudaMemsetAsync(cb, 0xff, 3 * 4, st));   // min of the centroids: from the largest key
    RT_CUDA(ctx, cudaMemsetAsync(cb + 3, 0, 3 * 4, st));  // max: from the smallest
    const int grid = (n + 255) / 256;
    bvh_leaf_boxes<<<grid, 256, 0, st>>>(in, n, ctx->win_lo, ctx->win_hi, boxes, cb);
    if (n == 1) {
        bvh_single_leaf<<<1, 32, 0, st>>>(boxes, d.bvh_nodes, depth);
    } else {
        unsigned long long* code = (unsigned long long*)(S + o_code);
        unsigned long long* code2 = (unsigned long long*)(S + o_code2);
        int* leaf = (int*)(S + o_leaf);
        int* leaf2 = (int*)(S + o_leaf2);
        int* parent = (int*)(S + o_par);
        bvh_morton<<<grid, 256, 0, st>>>(boxes, n, cb, code, leaf);
        RT_CUDA(ctx, cub::DeviceRadixSort::SortPairs(S + o_sort, sort_bytes, code, code2, leaf, leaf2, n, 0, 3 * (int)kMortonAxisBits, st));
        RT_CUDA(ctx, cudaMemsetAsync(S + o_arr, 0, (size_t)n_nodes * 4, st));
        bvh_hierarchy<<<(n - 1 + 255) / 256, 256, 0, st>>>(code2, leaf2, n, d.bvh_nodes, parent);
        bvh_fit<<<grid, 256, 0, st>>>(boxes, parent, n, d.bvh_nodes, (unsigned*)(S + o_arr), (int*)(S + o_h), depth);
    }
    RT_CUDA(ctx, cudaGetLastError());
    RT_CUDA(ctx, cudaMemcpyAsync(d.h_bvh_depth, depth, sizeof(int), cudaMemcpyDeviceToHost, st));
    RT_CUDA(ctx, cudaEventRecord(d.ev_b1, st));
    d.sc.bvh_nodes = n_nodes;
    return RT_OK;
}

// Listed leaves from which the automatic choice (option bvh_build = 1) builds the tree on the device.  Measured on a B200
// (profiles/r03_bvh_build.txt, DESIGN §7): from 1 003 leaves up the device tree gives the shorter time to image (C5 shape,
// 1 k - 1 M leaves: its build is shorter and its frames too); on C2's 485 leaves the host tree renders 0.6 ms faster while
// either build takes 0.1 ms.
constexpr int kBvhDeviceMinLeaves = 1000;

// RT_ACCEL_BVH: (re)build the tree when the scene or the movers' window changed.  The device build runs on every device
// of the context at once; a tree deeper than bvh_closest's stack allows is never published — the host build (median
// splits, depth ~log2 n) replaces it.
int ensure_bvh(rt_ctx* ctx) {
    if (!ctx->bvh_dirty) return RT_OK;
    const int mode = ctx->opt.bvh_build;
    const bool on_device = mode == 2 || (mode == 1 && ctx->n_list >= kBvhDeviceMinLeaves);
    bool too_deep = false;
    if (on_device) {
        for (auto& d : ctx->devs)
            if (int rc = bvh_enqueue_device(ctx, d)) return rc;
        for (auto& d : ctx->devs) {
            RT_CUDA(ctx, cudaSetDevice(d.dev));
            RT_CUDA(ctx, cudaStreamSynchronize(d.stream));
            float ms = 0.f;
            RT_CUDA(ctx, cudaEventElapsedTime(&ms, d.ev_b0, d.ev_b1));
            d.sc.bvh = d.bvh_nodes;
            d.bvh_builder = 1;
            d.bvh_depth = *d.h_bvh_depth;
            d.bvh_build_ns = (long long)((double)ms * 1e6);
            too_deep |= d.bvh_depth > kBvhMaxDepth;
        }
        cudaSetDevice(ctx->devs[0].dev);
    }
    if (!on_device || too_deep)
        if (int rc = bvh_build_host(ctx)) return rc;
    ctx->bvh_dirty = false;
    return RT_OK;
}

int ensure_stage(rt_ctx* ctx, DeviceBuffers& d, size_t bytes) {
    if (d.h_stage_bytes >= bytes) return RT_OK;
    if (d.h_stage) cudaFreeHost(d.h_stage);
    d.h_stage = nullptr;
    d.h_stage_bytes = 0;
    RT_CUDA(ctx, cudaHostAlloc(&d.h_stage, bytes, cudaHostAllocDefault));
    d.h_stage_bytes = bytes;
    return RT_OK;
}

// dlopen libnccl.so.2 (the system library, or the one a host process such as PyTorch already loaded) and build one
// communicator per device of the context.  Failing to do so is an error: the caller asked for the NCCL reduce.
int ensure_nccl(rt_ctx* ctx) {
    NcclApi& N = ctx->nccl;
    if (!N.comms.empty()) return RT_OK;
    if (!N.handle) {
        N.handle = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!N.handle) return fail(ctx, RT_ERR_NCCL, std::string("dlopen(libnccl.so.2): ") + dlerror());
        auto sym = [&](const char* name) { return dlsym(N.handle, name); };
        N.CommInitAll = (decltype(N.CommInitAll))sym("ncclCommInitAll");
        N.CommDestroy = (decltype(N.CommDestroy))sym("ncclCommDestroy");
        N.Reduce = (decltype(N.Reduce))sym("ncclReduce");
        N.GroupStart = (decltype(N.GroupStart))sym("ncclGroupStart");
        N.GroupEnd = (decltype(N.GroupEnd))sym("ncclGroupEnd");
        N.GetErrorString = (decltype(N.GetErrorString))sym("ncclGetErrorString");
        if (!N.CommInitAll || !N.CommDestroy || !N.Reduce || !N.GroupStart || !N.GroupEnd || !N.GetErrorString)
            return fail(ctx, RT_ERR_NCCL, "libnccl.so.2 lacks a required symbol");
    }
    std::vector<int> ids;
    for (auto& d : ctx->devs) ids.push_back(d.dev);
    N.comms.assign(ids.size(), nullptr);
    ncclResult_t r = N.CommInitAll(N.comms.data(), (int)ids.size(), ids.data());
    if (r != ncclSuccess) {
        N.comms.clear();
        return fail(ctx, RT_ERR_NCCL, std::string("ncclCommInitAll: ") + N.GetErrorString(r));
    }
    cudaSetDevice(ctx->devs[0].dev);
    return RT_OK;
}

int check_ready(rt_ctx* ctx) {
    if (!ctx) return RT_ERR_ARG;
    if (!ctx->has_scene) return fail(ctx, RT_ERR_STATE, "rt_set_scene has not been called");
    return RT_OK;
}

int check_camera_times(rt_ctx* ctx) {
    if (!ctx->has_cam) return fail(ctx, RT_ERR_STATE, "rt_set_camera has not been called");
    int rc = ctx->cam.type == CAM_THIN_LENS ? ensure_window(ctx, std::min(ctx->cam.t0, ctx->cam.t1), std::max(ctx->cam.t0, ctx->cam.t1))
                                            : ensure_window(ctx, 0.0, 0.0);
    if (rc) return rc;
    return ctx->accel == RT_ACCEL_BVH ? ensure_bvh(ctx) : RT_OK;
}

// Byte offsets of the scene blob's sections: one layout for rt_set_scene_ex and rt_set_scene_device, so that both write the
// same bytes.  Every section starts on a 256-byte boundary and takes at least 16 bytes.
struct SceneLayout {
    size_t cull_a, cull_tc, tc_row, c0r, c1, t0t1, orig, cull_of, flags, mat, mtype, mparam, mtex, srec, scol, tie, ttype, tparam,
        tchild, ptype, pq, paux, pxf, xops, xp, pvec, pperm, iwh, ioff, irgb;
    size_t bytes;
};

SceneLayout scene_layout(int n, int n_total, int n_cull, int n_direct, int tc_tiles, int nm_, int nt, int nxf, bool uses_perlin,
                         int n_img, size_t img_bytes) {
    SceneLayout L{};
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + std::max<size_t>(bytes, 16), 256); return o; };
    L.cull_a = take((size_t)(n_cull + n_direct) * 16);
    L.cull_tc = take((size_t)tc_tiles * tc::B_TILE_BYTES); L.tc_row = take((size_t)tc_tiles * tc::TILE_N * 4);
    L.c0r = take((size_t)n_total * 16); L.c1 = take((size_t)n_total * 16); L.t0t1 = take((size_t)n_total * 8);
    L.orig = take((size_t)n * 4); L.cull_of = take((size_t)n * 4); L.flags = take((size_t)n_total * 4); L.mat = take((size_t)n_total * 4);
    L.mtype = take((size_t)nm_ * 4); L.mparam = take((size_t)nm_ * 4); L.mtex = take((size_t)nm_ * 4);
    L.srec = take((size_t)n * 16); L.scol = take((size_t)n * 16); L.tie = take((size_t)n * 4);
    L.ttype = take((size_t)std::max(nt, 1) * 4); L.tparam = take((size_t)std::max(nt, 1) * 48); L.tchild = take((size_t)std::max(nt, 1) * 8);
    L.ptype = take((size_t)n_total * 4); L.pq = take((size_t)n_total * 48); L.paux = take((size_t)n_total * 8); L.pxf = take((size_t)n_total * 4);
    L.xops = take((size_t)nxf * RT_XFORM_MAX_OPS * 4); L.xp = take((size_t)nxf * RT_XFORM_MAX_OPS * 16);
    L.pvec = take(uses_perlin ? 256 * 16 : 0); L.pperm = take(uses_perlin ? 768 * 4 : 0);
    L.iwh = take((size_t)n_img * 8); L.ioff = take((size_t)n_img * 8); L.irgb = take(img_bytes);
    L.bytes = off;
    return L;
}

// the device's scene pointers into its blob
void set_dev_scene(DeviceBuffers& d, const SceneLayout& L, int n, int n_list, int n_cull, int tc_tiles, int generic, int n_total) {
    char* b = (char*)d.scene_blob;
    DevScene& sc = d.sc;
    sc = DevScene{};
    sc.n = n;
    sc.n_list = n_list;
    sc.n_cull = n_cull;
    sc.cull_a = (const float4*)(b + L.cull_a);
    sc.cull_tc = (const float*)(b + L.cull_tc);
    sc.tc_row_k = (const int*)(b + L.tc_row);
    sc.tc_tiles = tc_tiles;
    sc.ex_c0r = (const float4*)(b + L.c0r); sc.ex_c1 = (const float4*)(b + L.c1); sc.ex_t0t1 = (const float2*)(b + L.t0t1);
    sc.orig_id = (const int*)(b + L.orig); sc.cull_of_orig = (const int*)(b + L.cull_of);
    sc.flags = (const unsigned*)(b + L.flags); sc.mat_id = (const int*)(b + L.mat);
    sc.shade_rec = (const int4*)(b + L.srec); sc.shade_col = (const float4*)(b + L.scol);
    sc.mat_type = (const int*)(b + L.mtype); sc.mat_param = (const float*)(b + L.mparam); sc.mat_tex = (const int*)(b + L.mtex);
    sc.tex_type = (const int*)(b + L.ttype); sc.tex_params = (const float*)(b + L.tparam); sc.tex_child = (const int*)(b + L.tchild);
    sc.generic = generic;
    sc.n_total = n_total;
    sc.tie_hi = (const unsigned*)(b + L.tie);
    sc.prim_type = (const int*)(b + L.ptype); sc.prim_q = (const float4*)(b + L.pq); sc.prim_aux = (const int2*)(b + L.paux);
    sc.prim_xform = (const int*)(b + L.pxf); sc.xform_ops = (const int*)(b + L.xops); sc.xform_p = (const float4*)(b + L.xp);
    sc.perlin_vec = (const float4*)(b + L.pvec); sc.perlin_perm = (const int*)(b + L.pperm);
    sc.image_wh = (const int2*)(b + L.iwh); sc.image_off = (const long long*)(b + L.ioff); sc.image_rgb = (const unsigned char*)(b + L.irgb);
}

// a device blob of at least `bytes` (and its pinned staging copy), reused by the next upload
int ensure_scene_blob(rt_ctx* ctx, DeviceBuffers& d, size_t bytes) {
    if (d.scene_bytes >= bytes) return RT_OK;
    if (d.scene_blob) cudaFree(d.scene_blob);
    if (d.scene_stage) cudaFreeHost(d.scene_stage);
    d.scene_blob = nullptr; d.scene_stage = nullptr; d.scene_bytes = 0;
    const size_t cap = align_up(bytes + bytes / 4, 4096);
    RT_CUDA(ctx, cudaMalloc(&d.scene_blob, cap));
    RT_CUDA(ctx, cudaHostAlloc(&d.scene_stage, cap, cudaHostAllocDefault));
    d.scene_bytes = cap;
    return RT_OK;
}

}  // namespace

extern "C" {

int rt_abi_version(void) { return RT_ABI_VERSION; }

const char* rt_last_error(const rt_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int rt_create(rt_ctx** out, const int* device_ids, int n_devices) {
    if (!out) return fail(nullptr, RT_ERR_ARG, "out is null");
    *out = nullptr;
    if (n_devices < 0 || n_devices > 8) return fail(nullptr, RT_ERR_ARG, "n_devices must be in [1, 8]");
    if (n_devices == 0 || !device_ids) n_devices = 1;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(nullptr, RT_ERR_NODEVICE,
                    std::string("no usable CUDA device (") + cudaGetErrorString(e) + "); there is no CPU fallback");
    rt_ctx* ctx = new rt_ctx();
    ctx->opt = options_from_env();
    ctx->devs.resize(n_devices);
    ctx->peer_ok.assign(n_devices, false);
    for (int i = 0; i < n_devices; ++i) {
        DeviceBuffers& d = ctx->devs[i];
        d.dev = device_ids ? device_ids[i] : 0;
        if (d.dev < 0 || d.dev >= count) {
            g_create_error = "device id out of range";
            delete ctx;
            return RT_ERR_ARG;
        }
        cudaDeviceProp prop;
        if ((e = cudaSetDevice(d.dev)) != cudaSuccess || (e = cudaGetDeviceProperties(&prop, d.dev)) != cudaSuccess ||
            (e = cudaStreamCreateWithFlags(&d.stream, cudaStreamNonBlocking)) != cudaSuccess ||
            (e = cudaEventCreate(&d.ev0)) != cudaSuccess || (e = cudaEventCreate(&d.ev1)) != cudaSuccess ||
            (e = cudaEventCreateWithFlags(&d.ev_done, cudaEventDisableTiming)) != cudaSuccess ||
            (e = cudaEventCreate(&d.ev_r0)) != cudaSuccess || (e = cudaEventCreate(&d.ev_r1)) != cudaSuccess ||
            (e = cudaMalloc(&d.d_counters, (DC_COUNT + 1) * sizeof(unsigned long long))) != cudaSuccess ||
            (e = cudaMemset(d.d_counters, 0, (DC_COUNT + 1) * sizeof(unsigned long long))) != cudaSuccess) {
            g_create_error = std::string("device init: ") + cudaGetErrorString(e);
            rt_destroy(ctx);
            return RT_ERR_CUDA;
        }
        if (prop.major < 10) {
            g_create_error = std::string("device ") + prop.name + " is not sm_100-class; this library is sm_100a only";
            rt_destroy(ctx);
            return RT_ERR_NODEVICE;
        }
        d.sm_count = prop.multiProcessorCount;
        int khz = 0;
        cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, d.dev);
        d.clock_khz = khz;
        snprintf(d.name, sizeof(d.name), "%s", prop.name);
    }
    // peer access from the root device to every other device (NVLink loads in the reduce kernel)
    for (int i = 1; i < n_devices; ++i) {
        int can = 0;
        cudaDeviceCanAccessPeer(&can, ctx->devs[0].dev, ctx->devs[i].dev);
        if (can) {
            cudaSetDevice(ctx->devs[0].dev);
            cudaError_t pe = cudaDeviceEnablePeerAccess(ctx->devs[i].dev, 0);
            if (pe == cudaSuccess || pe == cudaErrorPeerAccessAlreadyEnabled) ctx->peer_ok[i] = true;
            cudaGetLastError();
        }
    }
    cudaSetDevice(ctx->devs[0].dev);
    *out = ctx;
    return RT_OK;
}

void rt_destroy(rt_ctx* ctx) {
    if (!ctx) return;
    for (auto c : ctx->nccl.comms)
        if (c && ctx->nccl.CommDestroy) ctx->nccl.CommDestroy(c);
    ctx->nccl.comms.clear();
    for (auto& d : ctx->devs) {
        cudaSetDevice(d.dev);
        if (d.stream) cudaStreamSynchronize(d.stream);
        if (d.scene_blob) cudaFree(d.scene_blob);
        if (d.scene_stage) cudaFreeHost(d.scene_stage);
        if (d.d_sum) cudaFree(d.d_sum);
        if (d.d_mean) cudaFree(d.d_mean);
        if (d.d_rgb8) cudaFree(d.d_rgb8);
        if (d.d_counters) cudaFree(d.d_counters);
        if (d.scratch) cudaFree(d.scratch);
        free_wave(d);
        if (d.ev0) cudaEventDestroy(d.ev0);
        if (d.ev1) cudaEventDestroy(d.ev1);
        if (d.ev_done) cudaEventDestroy(d.ev_done);
        if (d.ev_r0) cudaEventDestroy(d.ev_r0);
        if (d.ev_r1) cudaEventDestroy(d.ev_r1);
        for (auto& e : d.ev_chunk) if (e) cudaEventDestroy(e);
        if (d.h_stage) cudaFreeHost(d.h_stage);
        if (d.bvh_nodes) cudaFree(d.bvh_nodes);
        if (d.bvh_scratch) cudaFree(d.bvh_scratch);
        if (d.h_bvh_depth) cudaFreeHost(d.h_bvh_depth);
        if (d.bs_buf) cudaFree(d.bs_buf);
        if (d.sb_scratch) cudaFree(d.sb_scratch);
        if (d.h_sb) cudaFreeHost(d.h_sb);
        if (d.ev_sb) cudaEventDestroy(d.ev_sb);
        if (d.ev_b0) cudaEventDestroy(d.ev_b0);
        if (d.ev_b1) cudaEventDestroy(d.ev_b1);
        if (d.stream) cudaStreamDestroy(d.stream);
    }
    delete ctx;
}

int rt_device_info(rt_ctx* ctx, int* sm_count, int* clock_khz, char name[64]) {
    if (!ctx) return RT_ERR_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (sm_count) *sm_count = ctx->devs[0].sm_count;
    if (clock_khz) *clock_khz = ctx->devs[0].clock_khz;
    if (name) memcpy(name, ctx->devs[0].name, 64);
    return RT_OK;
}

// a point carried out of a leaf's wrapper chain (object space -> world), the way the hit point travels
// (hitable.clj:398-400, :443-449): last op first
static void xform_point_back(const rt_scene_ext* x, int xf, double p[3]) {
    if (xf < 0) return;
    int nops = 0;
    while (nops < RT_XFORM_MAX_OPS && x->xform_ops[RT_XFORM_MAX_OPS * xf + nops] != RT_XOP_NONE) ++nops;
    for (int q = nops - 1; q >= 0; --q) {
        const float* pr = x->xform_params + 4 * (size_t)(RT_XFORM_MAX_OPS * xf + q);
        const int op = x->xform_ops[RT_XFORM_MAX_OPS * xf + q];
        if (op == RT_XOP_TRANSLATE) { p[0] += pr[0]; p[1] += pr[1]; p[2] += pr[2]; }
        else if (op == RT_XOP_ROTATE_Y) {
            const double sn = pr[0], cs = pr[1], px = p[0], pz = p[2];
            p[0] = cs * px + sn * pz;
            p[2] = -(sn * px) + cs * pz;
        }
    }
}

// object-space bounding sphere of leaf i (caller's index): centre at t0 / t1, radius.  Media: see below.
static void leaf_bounds(const rt_scene_desc* s, const rt_scene_ext* x, int i, double c0[3], double c1[3], double* r) {
    const int type = (x && x->prim_type) ? x->prim_type[i] : RT_PRIM_SPHERE;
    const float* q = (x && x->prim_params) ? x->prim_params + 12 * (size_t)i : nullptr;
    if (type == RT_PRIM_SPHERE) {
        const bool moving = s->sphere_flags && (s->sphere_flags[i] & RT_SPHERE_MOVING) && s->center1 && s->t0t1;
        for (int c = 0; c < 3; ++c) {
            c0[c] = s->center0_r[4 * i + c];
            c1[c] = moving ? s->center1[4 * i + c] : c0[c];
        }
        *r = std::fabs((double)s->center0_r[4 * i + 3]);
    } else if (type == RT_PRIM_TRIANGLE) {
        double lo[3], hi[3];
        for (int c = 0; c < 3; ++c) {
            lo[c] = std::min({(double)q[c], (double)q[3 + c], (double)q[6 + c]});
            hi[c] = std::max({(double)q[c], (double)q[3 + c], (double)q[6 + c]});
            c0[c] = c1[c] = 0.5 * (lo[c] + hi[c]);
        }
        double r2 = 0.0;
        for (int v = 0; v < 3; ++v) {
            double d2 = 0.0;
            for (int c = 0; c < 3; ++c) d2 += (q[3 * v + c] - c0[c]) * (q[3 * v + c] - c0[c]);
            r2 = std::max(r2, d2);
        }
        *r = std::sqrt(r2) * (1.0 + 1e-6) + 1e-6;
    } else {   // rectangles: q = a0 b0 a1 b1 k
        const int axis = type == RT_PRIM_RECT_XY ? 2 : (type == RT_PRIM_RECT_XZ ? 1 : 0);
        const int A = type == RT_PRIM_RECT_YZ ? 1 : 0, B = type == RT_PRIM_RECT_XY ? 1 : 2;
        c0[A] = 0.5 * ((double)q[0] + q[2]); c0[B] = 0.5 * ((double)q[1] + q[3]); c0[axis] = q[4];
        for (int c = 0; c < 3; ++c) c1[c] = c0[c];
        const double da = 0.5 * ((double)q[2] - q[0]), db = 0.5 * ((double)q[3] - q[1]);
        *r = std::sqrt(da * da + db * db) * (1.0 + 1e-6) + 1e-6;
    }
}

// the material and texture tables of a scene (rt_set_scene_ex; x = null: rt_set_scene and rt_set_scene_device)
static int check_tables(rt_ctx* ctx, const rt_scene_desc* s, const rt_scene_ext* x, bool* uses_perlin) {
    const int nm_ = s->n_materials, nt = s->n_textures;
    if (nm_ <= 0 || !s->mat_type || !s->mat_param || !s->mat_tex) return fail(ctx, RT_ERR_ARG, "material table missing");
    if (nt < 0 || (nt > 0 && (!s->tex_type || !s->tex_params || !s->tex_children)))
        return fail(ctx, RT_ERR_ARG, "texture table missing");
    const int max_tex = x ? RT_TEX_IMAGE_MAP : RT_TEX_CHECKERBOARD, max_mat = x ? RT_MAT_ISOTROPIC : RT_MAT_DIFFUSE_LIGHT;
    for (int t = 0; t < nt; ++t) {
        int ty = s->tex_type[t];
        if (ty < RT_TEX_CONSTANT || ty > max_tex)
            return fail(ctx, RT_ERR_UNSUPPORTED, x ? "unknown texture type" : "texture type needs rt_set_scene_ex (texture.clj:60-138)");
        const int n_children = ty == RT_TEX_CHECKERBOARD ? 2 : ((ty == RT_TEX_FLIP_U || ty == RT_TEX_FLIP_V) ? 1 : 0);
        for (int c = 0; c < n_children; ++c) {
            int ch = s->tex_children[2 * t + c];
            if (ch < 0 || ch >= t) return fail(ctx, RT_ERR_ARG, "a texture's child must be an earlier texture id");
        }
        if (ty == RT_TEX_PERLIN_NOISE || ty == RT_TEX_PERLIN_TURB || ty == RT_TEX_MARBLE) *uses_perlin = true;
        if (ty == RT_TEX_IMAGE_MAP) {
            const int im = (int)s->tex_params[12 * t];
            if (im < 0 || im >= x->n_images || !x->image_wh || !x->image_offset || !x->image_rgb || x->image_wh[2 * im] <= 0 ||
                x->image_wh[2 * im + 1] <= 0)
                return fail(ctx, RT_ERR_ARG, "image texture refers to a missing image");
        }
    }
    if (*uses_perlin && (!x->perlin_vectors || !x->perlin_perm)) return fail(ctx, RT_ERR_ARG, "Perlin textures need the marshalled tables (perlin.clj:6-17)");
    for (int m = 0; m < nm_; ++m) {
        int ty = s->mat_type[m];
        if (ty < RT_MAT_LAMBERTIAN || ty > max_mat)
            return fail(ctx, RT_ERR_UNSUPPORTED, x ? "unknown material type" : "material type needs rt_set_scene_ex (shader.clj:129-143)");
        if (ty != RT_MAT_DIELECTRIC && (s->mat_tex[m] < 0 || s->mat_tex[m] >= nt))
            return fail(ctx, RT_ERR_ARG, "material texture id out of range");
    }
    return RT_OK;
}

// Upload: validate, reorder to cull order (listed leaves, then the "direct" spheres), build the FP32 cull
// records with their conservative inflation, and copy one blob per device.
int rt_set_scene_ex(rt_ctx* ctx, const rt_scene_desc* s, const rt_scene_ext* x) {
    if (!ctx) return RT_ERR_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (!s) return fail(ctx, RT_ERR_ARG, "scene is null");
    if (x && x->struct_bytes != (int32_t)sizeof(rt_scene_ext)) return fail(ctx, RT_ERR_ARG, "rt_scene_ext.struct_bytes does not match this library (ABI 2: 120 bytes)");
    const int n = s->n_spheres, nm_ = s->n_materials, nt = s->n_textures;
    const int nb = x ? x->n_boundary : 0, n_total = n + nb;
    if (n <= 0 || !s->center0_r || !s->material_id) return fail(ctx, RT_ERR_ARG, "scene needs at least one primitive");
    if (nb < 0) return fail(ctx, RT_ERR_ARG, "n_boundary is negative");
    bool uses_perlin = false;
    if (int rc = check_tables(ctx, s, x, &uses_perlin)) return rc;
    const int tie_rule = x ? x->tie_rule : RT_TIE_HITLIST;
    if (tie_rule != RT_TIE_HITLIST && tie_rule != RT_TIE_BVH) return fail(ctx, RT_ERR_ARG, "unknown tie rule");
    int generic = uses_perlin ? 1 : 0;
    for (int t = 0; t < nt; ++t) if (s->tex_type[t] > RT_TEX_CHECKERBOARD) generic = 1;
    for (int m = 0; m < nm_; ++m) if (s->mat_type[m] == RT_MAT_ISOTROPIC) generic = 1;
    if (x && (x->prim_type || x->prim_xform)) {
        if ((x->prim_type && !x->prim_params) || (x->n_xforms > 0 && (!x->xform_ops || !x->xform_params)) || x->n_xforms < 0)
            return fail(ctx, RT_ERR_ARG, "primitive / transform tables missing");
        for (int i = 0; i < n_total; ++i) {
            const int ty = x->prim_type ? x->prim_type[i] : RT_PRIM_SPHERE;
            if (ty < RT_PRIM_SPHERE || ty > RT_PRIM_MEDIUM) return fail(ctx, RT_ERR_UNSUPPORTED, "unknown primitive type");
            const int xf = x->prim_xform ? x->prim_xform[i] : -1;
            if (xf < -1 || xf >= x->n_xforms) return fail(ctx, RT_ERR_ARG, "transform index out of range");
            if (ty != RT_PRIM_SPHERE || xf >= 0) generic = 1;
            if (ty == RT_PRIM_MEDIUM) {
                if (i >= n) return fail(ctx, RT_ERR_ARG, "a medium cannot bound a medium");
                if (!x->prim_aux) return fail(ctx, RT_ERR_ARG, "prim_aux missing");
                const int first = x->prim_aux[2 * i], count = x->prim_aux[2 * i + 1];
                if (first < n || count < 1 || first + count > n_total) return fail(ctx, RT_ERR_ARG, "medium boundary out of range");
                if (!(x->prim_params[12 * (size_t)i] > 0.f)) return fail(ctx, RT_ERR_ARG, "medium density must be positive");
            }
        }
        for (int q = 0; q < x->n_xforms * RT_XFORM_MAX_OPS; ++q)
            if (x->xform_ops[q] < RT_XOP_NONE || x->xform_ops[q] > RT_XOP_FLIP) return fail(ctx, RT_ERR_UNSUPPORTED, "unknown transform op");
    } else if (nb > 0) {
        return fail(ctx, RT_ERR_ARG, "boundary primitives without a primitive table");
    }
    auto ptype = [&](int i) { return (x && x->prim_type) ? x->prim_type[i] : RT_PRIM_SPHERE; };
    double win_lo = INFINITY, win_hi = -INFINITY;
    for (int i = 0; i < n_total; ++i) {
        unsigned fl = s->sphere_flags ? s->sphere_flags[i] : 0u;
        if (ptype(i) != RT_PRIM_SPHERE) fl = 0u;
        bool moving = (fl & RT_SPHERE_MOVING) && s->center1 && s->t0t1;
        if (fl & ~(RT_SPHERE_UV | RT_SPHERE_MOVING)) return fail(ctx, RT_ERR_UNSUPPORTED, "unknown sphere flag");
        if (i < n && (s->material_id[i] < 0 || s->material_id[i] >= nm_)) return fail(ctx, RT_ERR_ARG, "material id out of range");
        if (moving) {
            double t0 = s->t0t1[2 * i], t1 = s->t0t1[2 * i + 1];
            if (!(t1 != t0)) return fail(ctx, RT_ERR_ARG, "moving sphere with t1 == t0");
            win_lo = std::min(win_lo, std::min(t0, t1));
            win_hi = std::max(win_hi, std::max(t0, t1));
        }
    }
    if (!(win_lo <= win_hi)) { win_lo = 0.0; win_hi = 0.0; }   // no movers
    if (ctx->has_cam) {                                           // cover the shutter interval already set
        double lo = ctx->cam.type == CAM_THIN_LENS ? std::min(ctx->cam.t0, ctx->cam.t1) : 0.0;
        double hi = ctx->cam.type == CAM_THIN_LENS ? std::max(ctx->cam.t0, ctx->cam.t1) : 0.0;
        win_lo = std::min(win_lo, lo);
        win_hi = std::max(win_hi, hi);
    }

    // Cull order: listed spheres first (caller's order), then the "direct" spheres that bypass the cull.  A sphere
    // is direct when it is large against the population (radius >= 8 x the median) and encloses or touches the
    // centroid of the small spheres (a sky dome, a ground sphere): nearly every ray starts inside it or on it, so
    // the cull would pass it anyway.  The choice changes the work split only — results are identical either way.
    std::vector<int> perm((size_t)n);
    int n_direct = 0;
    {
        std::vector<char> direct((size_t)n, 0);
        double direct_centroid[3] = {0, 0, 0};
        // Isotropic.scatter hands the hit's t to the scattered ray as its TIME (shader.clj:135, kept as written), so in a
        // scene with media a ray's time can leave every shutter window — and a MovingSphere is then met at an extrapolated
        // position no window-bound cull record covers.  There the movers bypass the cull / the tree and are tested exactly.
        bool any_iso = false;
        for (int m = 0; m < nm_; ++m) any_iso |= s->mat_type[m] == RT_MAT_ISOTROPIC;
        if (any_iso)
            for (int i = 0; i < n; ++i)
                if (ptype(i) == RT_PRIM_SPHERE && s->sphere_flags && (s->sphere_flags[i] & RT_SPHERE_MOVING) && s->center1 && s->t0t1) {
                    if (n_direct == 8) return fail(ctx, RT_ERR_UNSUPPORTED, "more than 8 moving spheres in a scene with Isotropic media");
                    direct[(size_t)i] = 1;
                    ++n_direct;
                }
        if (n_direct == n) { direct[0] = 0; --n_direct; }   // the cull list must not be empty
        if (n > 16 && ctx->opt.direct_spheres && !generic) {
            std::vector<double> radii((size_t)n);
            for (int i = 0; i < n; ++i) radii[(size_t)i] = std::fabs((double)s->center0_r[4 * i + 3]);
            std::vector<double> sorted = radii;
            std::nth_element(sorted.begin(), sorted.begin() + n / 2, sorted.end());
            const double big = 8.0 * sorted[(size_t)n / 2];
            double cen[3] = {0, 0, 0};
            int small = 0;
            for (int i = 0; i < n; ++i)
                if (radii[(size_t)i] < big) {
                    for (int c = 0; c < 3; ++c) cen[c] += s->center0_r[4 * i + c];
                    ++small;
                }
            for (int c = 0; c < 3; ++c) { cen[c] /= std::max(1, small); direct_centroid[c] = cen[c]; }
            std::vector<std::pair<double, int>> cand;
            for (int i = 0; i < n; ++i) {
                if (radii[(size_t)i] < big) continue;
                double d2 = 0.0;
                for (int c = 0; c < 3; ++c) { double xx = s->center0_r[4 * i + c] - cen[c]; d2 += xx * xx; }
                if (std::sqrt(d2) <= 1.05 * radii[(size_t)i]) cand.emplace_back(-radii[(size_t)i], i);
            }
            std::sort(cand.begin(), cand.end());
            for (size_t q = 0; q < cand.size() && q < 8; ++q) { direct[(size_t)cand[q].second] = 1; ++n_direct; }
        }
        int k = 0;
        for (int i = 0; i < n; ++i) if (!direct[(size_t)i]) perm[(size_t)k++] = i;
        // direct spheres: the ones whose surface passes near the population's centroid first (a ground sphere: a hit
        // there lets the distance pre-test skip the enclosing ones), the all-enclosing ones (a sky dome) last
        std::vector<std::pair<double, int>> order;
        for (int i = 0; i < n; ++i)
            if (direct[(size_t)i]) {
                double d2 = 0.0;
                for (int c = 0; c < 3; ++c) { double xx = s->center0_r[4 * i + c] - direct_centroid[c]; d2 += xx * xx; }
                order.emplace_back(-std::sqrt(d2) / std::max(1e-30, std::fabs((double)s->center0_r[4 * i + 3])), i);
            }
        std::sort(order.begin(), order.end());
        for (auto& o : order) perm[(size_t)k++] = o.second;
    }
    const int n_list = n - n_direct;
    const int n_cull = (int)align_up((size_t)n_list, CULL_PAD);
    // source index of entry k of the device arrays: world leaves in cull order, then the boundary leaves as given
    auto src = [&](int k) { return k < n ? perm[(size_t)k] : k; };

    // host copy of the geometry (cull order): the cull records are rebuilt when the time window has to grow
    ctx->h_c0r.assign(4 * (size_t)n_total, 0.f);
    ctx->h_c1.assign(4 * (size_t)n_total, 0.f);
    ctx->h_t0t1.assign(2 * (size_t)n_total, 0.f);
    ctx->h_flags.assign((size_t)n_total, 0u);
    ctx->h_bs_c0.assign(3 * (size_t)n, 0.0);
    ctx->h_bs_c1.assign(3 * (size_t)n, 0.0);
    ctx->h_bs_r.assign((size_t)n, 0.0);
    std::vector<int> h_mat((size_t)n_total, 0);
    for (int k = 0; k < n_total; ++k) {
        const int i = src(k);
        unsigned fl = (s->sphere_flags && ptype(i) == RT_PRIM_SPHERE) ? s->sphere_flags[i] : 0u;
        bool moving = (fl & RT_SPHERE_MOVING) && s->center1 && s->t0t1;
        ctx->h_flags[k] = moving ? fl : (fl & ~RT_SPHERE_MOVING);
        for (int c = 0; c < 4; ++c) ctx->h_c0r[4 * k + c] = s->center0_r[4 * i + c];
        for (int c = 0; c < 3; ++c) ctx->h_c1[4 * k + c] = moving ? s->center1[4 * i + c] : s->center0_r[4 * i + c];
        ctx->h_t0t1[2 * k] = moving ? s->t0t1[2 * i] : 0.f;
        ctx->h_t0t1[2 * k + 1] = moving ? s->t0t1[2 * i + 1] : 1.f;
        h_mat[(size_t)k] = k < n ? s->material_id[i] : 0;
    }
    // world-space bounding spheres of the world leaves (what the FP32 cull tests)
    for (int k = 0; k < n; ++k) {
        const int i = src(k);
        double c0[3], c1[3], r = 0.0;
        if (ptype(i) == RT_PRIM_MEDIUM) {
            // the sphere around its boundary leaves, each carried out of its own wrappers, then out of the medium's
            const int first = x->prim_aux[2 * i], count = x->prim_aux[2 * i + 1];
            std::vector<double> cs((size_t)count * 3), rs((size_t)count);
            double cen[3] = {0, 0, 0};
            for (int b = 0; b < count; ++b) {
                double b0[3], b1[3], br;
                leaf_bounds(s, x, first + b, b0, b1, &br);
                const int bxf = x->prim_xform ? x->prim_xform[first + b] : -1;
                xform_point_back(x, bxf, b0);
                xform_point_back(x, bxf, b1);
                double half = 0.0;
                for (int c = 0; c < 3; ++c) { cs[3 * (size_t)b + c] = 0.5 * (b0[c] + b1[c]); half += 0.25 * (b1[c] - b0[c]) * (b1[c] - b0[c]); cen[c] += cs[3 * (size_t)b + c] / count; }
                rs[(size_t)b] = br + std::sqrt(half);
            }
            for (int b = 0; b < count; ++b) {
                double d2 = 0.0;
                for (int c = 0; c < 3; ++c) d2 += (cs[3 * (size_t)b + c] - cen[c]) * (cs[3 * (size_t)b + c] - cen[c]);
                r = std::max(r, std::sqrt(d2) + rs[(size_t)b]);
            }
            for (int c = 0; c < 3; ++c) c0[c] = c1[c] = cen[c];
            r = r * (1.0 + 1e-6) + 1e-6;
        } else {
            leaf_bounds(s, x, i, c0, c1, &r);
        }
        const int xf = (x && x->prim_xform) ? x->prim_xform[i] : -1;
        if (xf >= 0) { xform_point_back(x, xf, c0); xform_point_back(x, xf, c1); r = r * (1.0 + 1e-6) + 1e-6 * (1.0 + std::fabs(c0[0]) + std::fabs(c0[1]) + std::fabs(c0[2])); }
        for (int c = 0; c < 3; ++c) { ctx->h_bs_c0[3 * (size_t)k + c] = c0[c]; ctx->h_bs_c1[3 * (size_t)k + c] = c1[c]; }
        ctx->h_bs_r[(size_t)k] = r;
    }
    ctx->n_list = n_list;
    ctx->n_cull = n_cull;
    ctx->n_spheres = n;
    ctx->n_total = n_total;
    ctx->generic = generic;

    const int tc_tiles = (n_list + tc::TILE_N - 1) / tc::TILE_N;   // (over MAX_TILES: several wf_cull_tc launches per iteration)
    ctx->tc_tiles = tc_tiles;
    ctx->bs_on_device = ctx->bs_mirror = false;
    {   // rows: the listed leaves dealt out over the 32-row words largest first (a leaf's share of the candidates grows with its
        // radius), so that every epilogue warp's columns see the same mix; the padding rows are spread the same way
        ctx->tc_row_k.assign((size_t)tc_tiles * tc::TILE_N, -1);
        ctx->tc_scratch_rows.assign((size_t)(tc_tiles ? n_list : 0), std::vector<float>());
        if (tc_tiles) {
            std::vector<int> order((size_t)n_list);
            for (int k = 0; k < n_list; ++k) order[(size_t)k] = k;
            std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return ctx->h_bs_r[(size_t)a] > ctx->h_bs_r[(size_t)b]; });
            const int words = tc_tiles * tc::TILE_N / 32;
            for (int i = 0; i < n_list; ++i) ctx->tc_row_k[(size_t)(i % words) * 32 + (size_t)(i / words)] = order[(size_t)i];
        }
    }
    const int nxf = x ? std::max(0, x->n_xforms) : 0;
    const int n_img = x ? std::max(0, x->n_images) : 0;
    size_t img_bytes = 0;
    for (int i = 0; i < n_img; ++i) img_bytes = std::max(img_bytes, (size_t)x->image_offset[i] + (size_t)x->image_wh[2 * i] * x->image_wh[2 * i + 1] * 3);
    const SceneLayout L = scene_layout(n, n_total, n_cull, n_direct, tc_tiles, nm_, nt, nxf, uses_perlin, n_img, img_bytes);
    const size_t o_cull_a = L.cull_a, o_cull_tc = L.cull_tc, o_tc_row = L.tc_row, o_c0r = L.c0r, o_c1 = L.c1, o_t0t1 = L.t0t1;
    const size_t o_orig = L.orig, o_cull_of = L.cull_of, o_flags = L.flags, o_mat = L.mat, o_mtype = L.mtype, o_mparam = L.mparam;
    const size_t o_mtex = L.mtex, o_srec = L.srec, o_scol = L.scol, o_tie = L.tie, o_ttype = L.ttype, o_tparam = L.tparam;
    const size_t o_tchild = L.tchild, o_ptype = L.ptype, o_pq = L.pq, o_paux = L.paux, o_pxf = L.pxf, o_xops = L.xops, o_xp = L.xp;
    const size_t o_pvec = L.pvec, o_pperm = L.pperm, o_iwh = L.iwh, o_ioff = L.ioff, o_irgb = L.irgb;
    std::vector<unsigned char> blob(L.bytes, 0);
    build_cull_records(ctx, win_lo, win_hi, (float*)(blob.data() + o_cull_a), tc_tiles ? (float*)(blob.data() + o_cull_tc) : nullptr);
    if (tc_tiles) memcpy(blob.data() + o_tc_row, ctx->tc_row_k.data(), ctx->tc_row_k.size() * 4);
    memcpy(blob.data() + o_c0r, ctx->h_c0r.data(), (size_t)n_total * 16);
    memcpy(blob.data() + o_c1, ctx->h_c1.data(), (size_t)n_total * 16);
    memcpy(blob.data() + o_t0t1, ctx->h_t0t1.data(), (size_t)n_total * 8);
    memcpy(blob.data() + o_flags, ctx->h_flags.data(), (size_t)n_total * 4);
    int* orig = (int*)(blob.data() + o_orig);
    int* cull_of = (int*)(blob.data() + o_cull_of);
    for (int k = 0; k < n; ++k) { orig[k] = perm[(size_t)k]; cull_of[perm[(size_t)k]] = k; }
    memcpy(blob.data() + o_mat, h_mat.data(), (size_t)n_total * 4);
    {   // per-leaf shading records (material and constant texture resolved once, here) and tie-break keys
        int* srec = (int*)(blob.data() + o_srec);
        float* scol = (float*)(blob.data() + o_scol);
        unsigned* tie = (unsigned*)(blob.data() + o_tie);
        for (int k = 0; k < n; ++k) {
            const int m = h_mat[(size_t)k], tex = s->mat_tex[m];
            const bool has_tex = s->mat_type[m] != RT_MAT_DIELECTRIC && tex >= 0 && tex < nt;
            const int tex_type = has_tex ? s->tex_type[tex] : -1;
            srec[4 * k + 0] = s->mat_type[m];
            srec[4 * k + 1] = tex;
            srec[4 * k + 2] = tex_type;
            srec[4 * k + 3] = (int)ctx->h_flags[(size_t)k];
            scol[4 * k + 0] = s->mat_param[m];
            for (int c = 0; c < 3; ++c) scol[4 * k + 1 + c] = tex_type == RT_TEX_CONSTANT ? s->tex_params[12 * tex + c] : 0.f;
            // exact ties in t (coincident geometry): the smallest key wins.  Hitlist world (hitable.clj:17-26): the first
            // strict-range leaf (sphere) in caller order, but a later inclusive-range leaf (rectangle / triangle / medium)
            // replaces an equal earlier hit; bvh-node world (hitable.clj:99-105, right child wins): the last leaf.
            const unsigned o_ = (unsigned)perm[(size_t)k];
            const bool strict = ptype(perm[(size_t)k]) == RT_PRIM_SPHERE;
            tie[k] = (tie_rule == RT_TIE_HITLIST && strict) ? (0x80000000u | o_) : (0x7fffffffu - o_);
        }
    }
    memcpy(blob.data() + o_mtype, s->mat_type, (size_t)nm_ * 4);
    memcpy(blob.data() + o_mparam, s->mat_param, (size_t)nm_ * 4);
    memcpy(blob.data() + o_mtex, s->mat_tex, (size_t)nm_ * 4);
    if (nt > 0) {
        memcpy(blob.data() + o_ttype, s->tex_type, (size_t)nt * 4);
        memcpy(blob.data() + o_tparam, s->tex_params, (size_t)nt * 48);
        memcpy(blob.data() + o_tchild, s->tex_children, (size_t)nt * 8);
    }
    if (generic) {
        int* pt = (int*)(blob.data() + o_ptype);
        float* pq = (float*)(blob.data() + o_pq);
        int* pa = (int*)(blob.data() + o_paux);
        int* pxf = (int*)(blob.data() + o_pxf);
        for (int k = 0; k < n_total; ++k) {
            const int i = src(k);
            pt[k] = ptype(i);
            if (x && x->prim_params) memcpy(pq + 12 * (size_t)k, x->prim_params + 12 * (size_t)i, 48);
            if (x && x->prim_aux) { pa[2 * k] = x->prim_aux[2 * i]; pa[2 * k + 1] = x->prim_aux[2 * i + 1]; }
            pxf[k] = (x && x->prim_xform) ? x->prim_xform[i] : -1;
        }
        if (nxf) {
            memcpy(blob.data() + o_xops, x->xform_ops, (size_t)nxf * RT_XFORM_MAX_OPS * 4);
            memcpy(blob.data() + o_xp, x->xform_params, (size_t)nxf * RT_XFORM_MAX_OPS * 16);
        }
    }
    if (uses_perlin) {
        float* pv = (float*)(blob.data() + o_pvec);
        for (int i = 0; i < 256; ++i)
            for (int c = 0; c < 3; ++c) pv[4 * i + c] = x->perlin_vectors[3 * i + c];
        memcpy(blob.data() + o_pperm, x->perlin_perm, 768 * 4);
    }
    if (n_img) {
        memcpy(blob.data() + o_iwh, x->image_wh, (size_t)n_img * 8);
        memcpy(blob.data() + o_ioff, x->image_offset, (size_t)n_img * 8);
        memcpy(blob.data() + o_irgb, x->image_rgb, img_bytes);
    }
    for (auto& d : ctx->devs) {
        RT_CUDA(ctx, cudaSetDevice(d.dev));
        RT_CUDA(ctx, cudaDeviceSynchronize());   // renders enqueued with sync = 0 on a caller's stream may still read the old scene
        if (int rc = ensure_scene_blob(ctx, d, blob.size())) return rc;
        memcpy(d.scene_stage, blob.data(), blob.size());
        RT_CUDA(ctx, cudaMemcpyAsync(d.scene_blob, d.scene_stage, blob.size(), cudaMemcpyHostToDevice, d.stream));
        RT_CUDA(ctx, cudaStreamSynchronize(d.stream));
        d.scene_used = blob.size();
        set_dev_scene(d, L, n, n_list, n_cull, tc_tiles, generic, n_total);
    }
    cudaSetDevice(ctx->devs[0].dev);
    // resident up to kTileCap records; beyond that the list is streamed through a smaller tile (tile_records,
    // a multiple of 512) so that several CTAs still fit on an SM
    const int tile_records = std::max(CHUNK, std::min(kTileCap, ctx->opt.tile_records / CHUNK * CHUNK));
    ctx->preloaded = n_cull <= kTileCap ? 1 : 0;
    ctx->cull_cap = ctx->preloaded ? std::max(n_cull, CULL_PAD) : tile_records;
    ctx->win_lo = win_lo;
    ctx->win_hi = win_hi;
    ctx->has_scene = true;
    ctx->bvh_dirty = true;
    return RT_OK;
}

int rt_set_scene(rt_ctx* ctx, const rt_scene_desc* s) { return rt_set_scene_ex(ctx, s, nullptr); }

// rt_set_scene with the per-primitive arrays in device memory: rt_set_scene_ex's steps for a sphere scene, run on the first
// device (rt_scene_build.cuh); the blob and the bounding spheres then go to every other device by peer copies.  Nothing but
// the tables and a small result crosses the host link.
int rt_set_scene_device(rt_ctx* ctx, const rt_scene_desc* s, void* stream) {
    if (!ctx) return RT_ERR_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (!s) return fail(ctx, RT_ERR_ARG, "scene is null");
    const int n = s->n_spheres, nm_ = s->n_materials, nt = s->n_textures;
    if (n <= 0 || !s->center0_r || !s->material_id) return fail(ctx, RT_ERR_ARG, "scene needs at least one primitive");
    bool uses_perlin = false;
    if (int rc = check_tables(ctx, s, nullptr, &uses_perlin)) return rc;
    DeviceBuffers& d0 = ctx->devs[0];
    RT_CUDA(ctx, cudaSetDevice(d0.dev));
    for (const void* p : {(const void*)s->center0_r, (const void*)s->center1, (const void*)s->t0t1, (const void*)s->sphere_flags,
                          (const void*)s->material_id}) {
        if (!p) continue;
        cudaPointerAttributes a{};
        const cudaError_t e = cudaPointerGetAttributes(&a, p);
        if (e != cudaSuccess) cudaGetLastError();   // not a pointer the runtime knows: clear the error, reject below
        if (e != cudaSuccess || (a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged) || a.device != d0.dev)
            return fail(ctx, RT_ERR_ARG, "rt_set_scene_device: a per-primitive array is not device memory on the context's first device");
    }

    // scratch of the first device: result | radii | sorted radii | partial sums | candidates | candidate count | cull order |
    // radius keys and leaf values of the feature-row sort (in, out) | cub storage
    const size_t n_ = (size_t)n;
    const bool want_direct = n > 16 && ctx->opt.direct_spheres;
    const cudaStream_t st = d0.stream;
    size_t sort_cap = 0;   // both sorts: (u64 key, int) pairs; radii are non-negative, so their bits sort as their values
    RT_CUDA(ctx, cub::DeviceRadixSort::SortPairs(nullptr, sort_cap, (const unsigned long long*)nullptr, (unsigned long long*)nullptr,
                                                 (const int*)nullptr, (int*)nullptr, n, 0, 64, st));
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off = align_up(off + bytes, 256); return o; };
    const size_t o_res = take(sizeof(SbResult)), o_rad = take(n_ * 8), o_sorted = take(n_ * 8), o_part = take((size_t)kSbPartials * 4 * 8);
    const size_t o_cand = take(n_ * 4), o_ncand = take(4), o_perm = take(n_ * 4), o_key = take(n_ * 8), o_key2 = take(n_ * 8);
    const size_t o_val = take(n_ * 4), o_val2 = take(n_ * 4), o_sort = take(sort_cap);
    if (d0.sb_scratch_bytes < off) {
        if (d0.sb_scratch) cudaFree(d0.sb_scratch);
        d0.sb_scratch = nullptr;
        d0.sb_scratch_bytes = 0;
        RT_CUDA(ctx, cudaMalloc(&d0.sb_scratch, off));
        d0.sb_scratch_bytes = off;
    }
    if (!d0.h_sb) {
        RT_CUDA(ctx, cudaHostAlloc((void**)&d0.h_sb, sizeof(SbResult), cudaHostAllocDefault));
        RT_CUDA(ctx, cudaEventCreateWithFlags(&d0.ev_sb, cudaEventDisableTiming));
    }
    char* W = (char*)d0.sb_scratch;
    SbResult* res = (SbResult*)(W + o_res);
    double* radii = (double*)(W + o_rad);
    double* sorted = (double*)(W + o_sorted);
    int* perm = (int*)(W + o_perm);
    const SbInput in{s->center0_r, s->center1, s->t0t1, s->sphere_flags, s->material_id, n, nm_};
    const int grid = (n + kSbBlock - 1) / kSbBlock;

    // 1. validation and the movers' window, 2. the direct spheres; one small read-back
    RT_CUDA(ctx, cudaEventRecord(d0.ev_sb, (cudaStream_t)stream));   // the caller's writes to the arrays come first
    RT_CUDA(ctx, cudaStreamWaitEvent(st, d0.ev_sb, 0));
    *d0.h_sb = SbResult{~0ull, 0xffffffffu, 0u, 0, {}, {}};
    RT_CUDA(ctx, cudaMemcpyAsync(res, d0.h_sb, sizeof(SbResult), cudaMemcpyHostToDevice, st));
    sb_validate<<<grid, kSbBlock, 0, st>>>(in, res, want_direct ? radii : nullptr);
    if (want_direct) {
        size_t sort_bytes = sort_cap;   // (the values are scratch: only the sorted radii are used)
        RT_CUDA(ctx, cub::DeviceRadixSort::SortPairs(W + o_sort, sort_bytes, (const unsigned long long*)radii, (unsigned long long*)sorted,
                                                     (const int*)(W + o_val), (int*)(W + o_val2), n, 0, 64, st));
        sb_small_partials<<<kSbPartials, kSbBlock, 0, st>>>(in, radii, sorted, (double*)(W + o_part));
        sb_centroid<<<1, kSbPartials, 0, st>>>((const double*)(W + o_part), res);
        RT_CUDA(ctx, cudaMemsetAsync(W + o_ncand, 0, 4, st));
        sb_candidates<<<grid, kSbBlock, 0, st>>>(in, radii, sorted, res, (int*)(W + o_cand), (unsigned*)(W + o_ncand));
        sb_direct_choose<<<1, 32, 0, st>>>(in, radii, (const int*)(W + o_cand), (const unsigned*)(W + o_ncand), res);
    }
    RT_CUDA(ctx, cudaGetLastError());
    RT_CUDA(ctx, cudaMemcpyAsync(d0.h_sb, res, sizeof(SbResult), cudaMemcpyDeviceToHost, st));
    RT_CUDA(ctx, cudaStreamSynchronize(st));
    const SbResult R = *d0.h_sb;
    if (R.err != ~0ull) {   // the first failing primitive, its first failing check: the host loop's error
        const int check = (int)(R.err & 3ull);
        if (check == 0) return fail(ctx, RT_ERR_UNSUPPORTED, "unknown sphere flag");
        return fail(ctx, RT_ERR_ARG, check == 1 ? "material id out of range" : "moving sphere with t1 == t0");
    }
    auto unordered = [](unsigned u) {
        u = (u & 0x80000000u) ? (u & 0x7fffffffu) : ~u;
        float f;
        memcpy(&f, &u, 4);
        return (double)f;
    };
    const bool any_moving = R.win_hi >= R.win_lo;
    double win_lo = any_moving ? unordered(R.win_lo) : 0.0, win_hi = any_moving ? unordered(R.win_hi) : 0.0;
    if (ctx->has_cam) {   // cover the shutter interval already set
        double lo = ctx->cam.type == CAM_THIN_LENS ? std::min(ctx->cam.t0, ctx->cam.t1) : 0.0;
        double hi = ctx->cam.type == CAM_THIN_LENS ? std::max(ctx->cam.t0, ctx->cam.t1) : 0.0;
        win_lo = std::min(win_lo, lo);
        win_hi = std::max(win_hi, hi);
    }
    const int n_direct = want_direct ? R.n_direct : 0;
    const int n_list = n - n_direct;
    const int n_cull = (int)align_up((size_t)n_list, CULL_PAD);
    const int tc_tiles = (n_list + tc::TILE_N - 1) / tc::TILE_N, rows = tc_tiles * tc::TILE_N;
    const SceneLayout L = scene_layout(n, n, n_cull, n_direct, tc_tiles, nm_, nt, 0, false, 0, 0);
    const size_t bs_bytes = n_ * 7 * 8;   // c0 [3n], c1 [3n], r [n]

    for (auto& d : ctx->devs) {
        RT_CUDA(ctx, cudaSetDevice(d.dev));
        RT_CUDA(ctx, cudaDeviceSynchronize());   // renders enqueued with sync = 0 on a caller's stream may still read the old scene
        if (int rc = ensure_scene_blob(ctx, d, L.bytes)) return rc;
        if (d.bs_bytes < bs_bytes) {
            if (d.bs_buf) cudaFree(d.bs_buf);
            d.bs_buf = nullptr;
            d.bs_bytes = 0;
            RT_CUDA(ctx, cudaMalloc(&d.bs_buf, bs_bytes));
            d.bs_bytes = bs_bytes;
        }
    }
    RT_CUDA(ctx, cudaSetDevice(d0.dev));
    ctx->n_list = n_list;
    ctx->n_cull = n_cull;
    ctx->n_spheres = n;
    ctx->n_total = n;
    ctx->generic = 0;
    ctx->tc_tiles = tc_tiles;
    ctx->tc_row_k.clear();
    ctx->tc_scratch_rows.clear();
    ctx->bs_on_device = true;
    ctx->bs_mirror = false;
    ctx->any_moving = any_moving;
    for (auto& d : ctx->devs) {
        set_dev_scene(d, L, n, n_list, n_cull, tc_tiles, 0, n);
        double* bs = (double*)d.bs_buf;
        d.bs_in = BvhLeafInput{bs, bs + 3 * n_, bs + 6 * n_, (const float*)d.sc.ex_t0t1, d.sc.flags};
        d.scene_used = L.bytes;
    }

    // 3. the blob, zeroed (the host's blob is a zero-filled vector), with the tables staged through pinned memory
    char* B = (char*)d0.scene_blob;
    char* S = (char*)d0.scene_stage;
    RT_CUDA(ctx, cudaMemsetAsync(B, 0, L.bytes, st));
    auto table = [&](size_t o, const void* src, size_t bytes) -> cudaError_t {
        memcpy(S + o, src, bytes);
        return cudaMemcpyAsync(B + o, S + o, bytes, cudaMemcpyHostToDevice, st);
    };
    RT_CUDA(ctx, table(L.mtype, s->mat_type, (size_t)nm_ * 4));
    RT_CUDA(ctx, table(L.mparam, s->mat_param, (size_t)nm_ * 4));
    RT_CUDA(ctx, table(L.mtex, s->mat_tex, (size_t)nm_ * 4));
    if (nt > 0) {
        RT_CUDA(ctx, table(L.ttype, s->tex_type, (size_t)nt * 4));
        RT_CUDA(ctx, table(L.tparam, s->tex_params, (size_t)nt * 48));
        RT_CUDA(ctx, table(L.tchild, s->tex_children, (size_t)nt * 8));
    }
    if (n_direct) sb_perm<<<grid, kSbBlock, 0, st>>>(n, res, perm);
    unsigned long long* key = (unsigned long long*)(W + o_key);
    int* val = (int*)(W + o_val);
    const SbBlob blob{(float*)(B + L.c0r), (float*)(B + L.c1), (float*)(B + L.t0t1), (unsigned*)(B + L.flags), (int*)(B + L.mat),
                      (int*)(B + L.orig), (int*)(B + L.cull_of), (int*)(B + L.srec), (float*)(B + L.scol), (unsigned*)(B + L.tie),
                      (const int*)(B + L.mtype), (const float*)(B + L.mparam), (const int*)(B + L.mtex), (const int*)(B + L.ttype),
                      (const float*)(B + L.tparam), nt, (double*)d0.bs_in.c0, (double*)d0.bs_in.c1, (double*)d0.bs_in.r, key, val, n_list};
    sb_gather<<<grid, kSbBlock, 0, st>>>(in, n_direct ? perm : nullptr, blob);
    // 4. the feature rows: listed leaves by bounding radius, descending, stable; dealt over the 32-row words
    size_t sort_bytes = 0;
    RT_CUDA(ctx, cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, (const unsigned long long*)nullptr, (unsigned long long*)nullptr,
                                                 (const int*)nullptr, (int*)nullptr, n_list, 0, 64, st));
    if (sort_bytes > sort_cap) return fail(ctx, RT_ERR_STATE, "rt_set_scene_device: sort storage underestimated");
    RT_CUDA(ctx, cub::DeviceRadixSort::SortPairs(W + o_sort, sort_bytes, key, (unsigned long long*)(W + o_key2), val, (int*)(W + o_val2),
                                                 n_list, 0, 64, st));
    sb_deal<<<(rows + kSbBlock - 1) / kSbBlock, kSbBlock, 0, st>>>((const int*)(W + o_val2), n_list, rows, (int*)(B + L.tc_row));
    RT_CUDA(ctx, cudaGetLastError());
    // 5. the cull records, the padding records and the rows' slots
    if (int rc = enqueue_records_device(ctx, d0, win_lo, win_hi)) return rc;
    // every other device: the same bytes
    for (size_t q = 1; q < ctx->devs.size(); ++q) {
        DeviceBuffers& d = ctx->devs[q];
        RT_CUDA(ctx, cudaMemcpyPeerAsync(d.scene_blob, d.dev, d0.scene_blob, d0.dev, L.bytes, st));
        RT_CUDA(ctx, cudaMemcpyPeerAsync(d.bs_buf, d.dev, d0.bs_buf, d0.dev, bs_bytes, st));
    }
    RT_CUDA(ctx, cudaStreamSynchronize(st));
    const int tile_records = std::max(CHUNK, std::min(kTileCap, ctx->opt.tile_records / CHUNK * CHUNK));
    ctx->preloaded = n_cull <= kTileCap ? 1 : 0;
    ctx->cull_cap = ctx->preloaded ? std::max(n_cull, CULL_PAD) : tile_records;
    ctx->win_lo = win_lo;
    ctx->win_hi = win_hi;
    ctx->has_scene = true;
    ctx->bvh_dirty = true;
    return RT_OK;
}

int rt_get_scene_blob(rt_ctx* ctx, int device_index, void* out, size_t cap, size_t* bytes) {
    if (!ctx) return RT_ERR_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (int rc = check_ready(ctx)) return rc;
    if (device_index < 0 || device_index >= (int)ctx->devs.size()) return fail(ctx, RT_ERR_ARG, "device_index out of range");
    const DeviceBuffers& d = ctx->devs[(size_t)device_index];
    if (bytes) *bytes = d.scene_used;
    if (out) {
        if (cap < d.scene_used) return fail(ctx, RT_ERR_ARG, "cap is below the blob's size (*bytes)");
        RT_CUDA(ctx, cudaSetDevice(d.dev));
        RT_CUDA(ctx, cudaMemcpy(out, d.scene_blob, d.scene_used, cudaMemcpyDeviceToHost));
        cudaSetDevice(ctx->devs[0].dev);
    }
    return RT_OK;
}

int rt_set_accel(rt_ctx* ctx, int accel) {
    if (!ctx) return RT_ERR_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (accel != RT_ACCEL_BRUTE_FORCE && accel != RT_ACCEL_BVH) return fail(ctx, RT_ERR_ARG, "unknown accelerator");
    ctx->accel = accel;
    if (accel == RT_ACCEL_BVH && ctx->has_scene) return ensure_bvh(ctx);
    return RT_OK;
}

int rt_get_bvh(rt_ctx* ctx, int device_index, float* out_nodes, int64_t cap_nodes, int64_t info[4]) {
    if (!ctx) return RT_ERR_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (int rc = check_ready(ctx)) return rc;
    if (device_index < 0 || device_index >= (int)ctx->devs.size()) return fail(ctx, RT_ERR_ARG, "device_index out of range");
    if (int rc = ensure_bvh(ctx)) return rc;
    DeviceBuffers& d = ctx->devs[(size_t)device_index];
    const int64_t n_nodes = d.sc.bvh_nodes;
    if (info) {
        info[0] = n_nodes;
        info[1] = d.bvh_depth;
        info[2] = d.bvh_builder;
        info[3] = d.bvh_build_ns;
    }
    if (out_nodes) {
        if (cap_nodes < n_nodes) return fail(ctx, RT_ERR_ARG, "cap_nodes is below the node count (info[0])");
        RT_CUDA(ctx, cudaSetDevice(d.dev));
        RT_CUDA(ctx, cudaMemcpy(out_nodes, d.bvh_nodes, (size_t)n_nodes * 4 * sizeof(float4), cudaMemcpyDeviceToHost));
        cudaSetDevice(ctx->devs[0].dev);
    }
    return RT_OK;
}

int rt_set_option(rt_ctx* ctx, const char* name, int64_t value) {
    if (!ctx) return RT_ERR_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (!name) return fail(ctx, RT_ERR_ARG, "option name is null");
    Options& o = ctx->opt;
    const std::string k(name);
    if (k == "wave_lanes") o.wave_lanes = (int)value;
    else if (k == "wave_capacity") o.wave_capacity = value;
    else if (k == "cull_claims") o.cull_claims = (int)value;
    else if (k == "cull_ctas_per_sm") o.cull_ctas_per_sm = (int)value;
    else if (k == "cull_shape") o.cull_shape = (int)value;
    else if (k == "light_block") o.light_block = (int)value;
    else if (k == "tail_entries") o.tail_entries = value;
    else if (k == "tail_ctas_per_sm") o.tail_ctas_per_sm = (int)value;
    else if (k == "tile_records") o.tile_records = (int)value;   // takes effect at the next rt_set_scene
    else if (k == "direct_spheres") o.direct_spheres = (int)value;   // takes effect at the next rt_set_scene
    else if (k == "common_origin") o.common_origin = (int)value;
    else if (k == "reduce") o.reduce = (int)value;
    else if (k == "rows") o.rows = (int)value;
    else if (k == "wave_depth") o.wave_depth = (int)value;
    else if (k == "mega_regcap") o.mega_regcap = (int)value;
    else if (k == "tail_rays") o.tail_rays = (int)value;
    else if (k == "tail_solo") o.tail_solo = (int)value;
    else if (k == "tail_lpp") o.tail_lpp = (int)value;
    else if (k == "tail_block") o.tail_block = (int)value;
    else if (k == "cull_tc") o.cull_tc = (int)value;
    else if (k == "tc_tiles_per_cta") o.tc_tiles_per_cta = (int)value;
    else if (k == "tc_ctas") o.tc_ctas = (int)value;
    else if (k == "bvh_build") o.bvh_build = (int)value;   // takes effect at the next tree build
    else return fail(ctx, RT_ERR_ARG, "unknown option: " + k);
    return RT_OK;
}

int rt_set_camera(rt_ctx* ctx, int cam_type, const float cam[24]) {
    if (!ctx) return RT_ERR_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (!cam) return fail(ctx, RT_ERR_ARG, "cam is null");
    if (cam_type != RT_CAM_PINHOLE && cam_type != RT_CAM_THIN_LENS) return fail(ctx, RT_ERR_UNSUPPORTED, "unknown camera type");
    DevCamera& c = ctx->cam;
    c.type = cam_type;
    auto g = [&](int k) { return make_float3(cam[3 * k], cam[3 * k + 1], cam[3 * k + 2]); };
    c.origin = g(0); c.lleft = g(1); c.horiz = g(2); c.vert = g(3); c.u = g(4); c.v = g(5); c.w = g(6);
    c.lens_radius = cam[21] / 2.0f;   // camera.clj:38
    c.t0 = cam[22];
    c.t1 = cam[23];
    ctx->has_cam = true;
    return RT_OK;
}

int rt_render_accumulate_device(rt_ctx* ctx, int nx, int ny, int sample_begin, int sample_count, int row_offset,
                                int row_stride, int max_depth, uint64_t seed, int variant, float* d_sum, void* stream,
                                int sync) {
    int rc = check_ready(ctx);
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if ((rc = check_camera_times(ctx))) return rc;
    if (nx <= 0 || ny <= 0 || sample_count < 0 || sample_begin < 0 || max_depth < 0 || !d_sum || row_stride < 1 ||
        row_offset < 0 || row_offset >= row_stride)
        return fail(ctx, RT_ERR_ARG, "bad render arguments");
    if ((long long)nx * ny > 0x7fffffffLL / 3) return fail(ctx, RT_ERR_ARG, "image too large");
    DeviceBuffers& d = ctx->devs[0];
    RT_CUDA(ctx, cudaSetDevice(d.dev));
    cudaStream_t st = (cudaStream_t)stream;
    RT_CUDA(ctx, cudaEventRecord(d.ev0, st));
    rc = launch_render(ctx, d, nx, ny, sample_begin, sample_count, row_offset, row_stride, max_depth, seed, variant, d_sum, st);
    if (rc) return rc;
    RT_CUDA(ctx, cudaEventRecord(d.ev1, st));
    d.timed = true;
    if (sync) RT_CUDA(ctx, cudaStreamSynchronize(st));
    return RT_OK;
}

int rt_resolve_device(rt_ctx* ctx, int nx, int ny, int nsamples_total, const float* d_sum, uint8_t* d_rgb8, void* stream,
                      int sync) {
    if (!ctx) return RT_ERR_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (nx <= 0 || ny <= 0 || nsamples_total <= 0 || !d_sum || !d_rgb8) return fail(ctx, RT_ERR_ARG, "bad resolve arguments");
    DeviceBuffers& d = ctx->devs[0];
    RT_CUDA(ctx, cudaSetDevice(d.dev));
    ResolveParams P{};
    P.sum = d_sum; P.n_peers = 0; P.nx = nx; P.ny = ny; P.nr = nsamples_total; P.rgb8 = d_rgb8; P.mean = nullptr; P.sum_out = nullptr;
    int total = nx * ny * 3;
    cudaStream_t st = (cudaStream_t)stream;
    resolve_kernel<<<(total + 255) / 256, 256, 0, st>>>(P);
    RT_CUDA(ctx, cudaGetLastError());
    ctx->n_launches += 1;
    if (sync) RT_CUDA(ctx, cudaStreamSynchronize(st));
    return RT_OK;
}

int rt_render(rt_ctx* ctx, int nx, int ny, int nsamples, int max_depth, uint64_t seed, int variant, float* out_linear_rgb,
              uint8_t* out_rgb8) {
    int rc = check_ready(ctx);
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if ((rc = check_camera_times(ctx))) return rc;
    if (nx <= 0 || ny <= 0 || nsamples <= 0 || max_depth < 0) return fail(ctx, RT_ERR_ARG, "bad render arguments");
    if ((long long)nx * ny > 0x7fffffffLL / 3) return fail(ctx, RT_ERR_ARG, "image too large");
    const size_t px = (size_t)nx * ny;
    const int G = (int)ctx->devs.size();
    const bool by_rows = G > 1 && ctx->opt.rows != 0;
    const bool use_nccl = G > 1 && ctx->opt.reduce != 0;
    if (use_nccl && (rc = ensure_nccl(ctx))) return rc;
    // Partition over the devices of the context (core.clj:100-108's chunk pool, SURVEY 8e): sample slices — device g
    // renders samples [g*S/G, (g+1)*S/G) of every pixel — or interleaved rows — device g renders rows j = g (mod G) with
    // all S samples.  One host thread per device (each feeds its own wavefront loop).
    auto device_work = [&](int g) -> int {
        DeviceBuffers& d = ctx->devs[g];
        RT_CUDA(ctx, cudaSetDevice(d.dev));
        int r = ensure_frame(ctx, d, px);
        if (r) return r;
        int s0 = (int)((long long)nsamples * g / G), s1 = (int)((long long)nsamples * (g + 1) / G);
        RT_CUDA(ctx, cudaEventRecord(d.ev0, d.stream));
        RT_CUDA(ctx, cudaMemsetAsync(d.d_sum, 0, px * 3 * sizeof(float), d.stream));
        if (by_rows) r = launch_render(ctx, d, nx, ny, 0, nsamples, g, G, max_depth, seed, variant, d.d_sum, d.stream);
        else r = launch_render(ctx, d, nx, ny, s0, s1 - s0, 0, 1, max_depth, seed, variant, d.d_sum, d.stream);
        if (r) return r;
        RT_CUDA(ctx, cudaEventRecord(d.ev1, d.stream));
        RT_CUDA(ctx, cudaEventRecord(d.ev_done, d.stream));
        d.timed = true;
        return RT_OK;
    };
    if (G == 1) {
        if ((rc = device_work(0))) return rc;
    } else {
        std::vector<int> rcs((size_t)G, RT_OK);
        std::vector<std::thread> workers;
        for (int g = 0; g < G; ++g) workers.emplace_back([&, g] { rcs[(size_t)g] = device_work(g); });
        for (auto& w : workers) w.join();
        int bad = RT_OK;
        for (int g = 0; g < G; ++g)
            if (rcs[(size_t)g] && !bad) bad = rcs[(size_t)g];
        if (bad) {   // the other devices may still be rendering into buffers the next call reuses: drain them first
            for (auto& dv : ctx->devs) { cudaSetDevice(dv.dev); cudaDeviceSynchronize(); }
            cudaSetDevice(ctx->devs[0].dev);
            return bad;
        }
    }
    // combine on the root device.  Default: the resolve kernel reads the peers' float sums over NVLink peer mappings (the
    // reduce fused into core.clj:52-57's gamma / quantise pass).  Option "reduce" = 1: one ncclReduce(sum, float32,
    // nx*ny*3, root 0) over the per-device communicators, then the plain resolve.
    DeviceBuffers& root = ctx->devs[0];
    RT_CUDA(ctx, cudaSetDevice(root.dev));
    ResolveParams P{};
    P.sum = root.d_sum; P.n_peers = 0; P.nx = nx; P.ny = ny; P.nr = nsamples;
    P.rgb8 = out_rgb8 ? root.d_rgb8 : nullptr;
    P.mean = out_linear_rgb ? root.d_mean : nullptr;
    P.sum_out = nullptr;
    const int total = nx * ny * 3;
    if (use_nccl) {
        NcclApi& N = ctx->nccl;
        for (int g = 1; g < G; ++g) RT_CUDA(ctx, cudaStreamWaitEvent(root.stream, ctx->devs[g].ev_done, 0));   // time the reduce alone
        RT_CUDA(ctx, cudaEventRecord(root.ev_r0, root.stream));
        ncclResult_t nr = N.GroupStart();
        for (int g = 0; g < G && nr == ncclSuccess; ++g)
            nr = N.Reduce(ctx->devs[g].d_sum, ctx->devs[g].d_sum, (size_t)total, ncclFloat, ncclSum, 0, N.comms[(size_t)g], ctx->devs[g].stream);
        const ncclResult_t ge = N.GroupEnd();
        if (nr == ncclSuccess) nr = ge;
        if (nr != ncclSuccess) {
            for (auto& dv : ctx->devs) { cudaSetDevice(dv.dev); cudaDeviceSynchronize(); }
            cudaSetDevice(root.dev);
            return fail(ctx, RT_ERR_NCCL, std::string("ncclReduce: ") + N.GetErrorString(nr));
        }
        RT_CUDA(ctx, cudaSetDevice(root.dev));
        RT_CUDA(ctx, cudaEventRecord(root.ev_r1, root.stream));
        resolve_kernel<<<(total + 255) / 256, 256, 0, root.stream>>>(P);
    } else {
        for (int g = 1; g < G; ++g) {
            DeviceBuffers& d = ctx->devs[g];
            RT_CUDA(ctx, cudaStreamWaitEvent(root.stream, d.ev_done, 0));
            if (ctx->peer_ok[g]) {
                P.peers[P.n_peers++] = d.d_sum;
            } else {   // no peer mapping: stage through a copy, then add
                if ((rc = ensure_scratch(ctx, root, (size_t)(G - 1) * px * 3 * sizeof(float)))) return rc;
                float* stage = (float*)root.scratch + (size_t)(g - 1) * px * 3;
                RT_CUDA(ctx, cudaMemcpyPeerAsync(stage, root.dev, d.d_sum, d.dev, px * 3 * sizeof(float), root.stream));
                P.peers[P.n_peers++] = stage;
            }
        }
        RT_CUDA(ctx, cudaEventRecord(root.ev_r0, root.stream));
        resolve_kernel<<<(total + 255) / 256, 256, 0, root.stream>>>(P);   // reduce + resolve in one pass
        RT_CUDA(ctx, cudaEventRecord(root.ev_r1, root.stream));
    }
    RT_CUDA(ctx, cudaGetLastError());
    ctx->n_launches += 1;
    // results: D2H into pinned staging at link speed, then one host memcpy into the caller's (pageable) buffer
    auto host_pinned = [](const void* p) {
        cudaPointerAttributes at{};
        if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
        return at.type == cudaMemoryTypeHost;
    };
    const size_t b_lin = out_linear_rgb ? align_up(px * 3 * sizeof(float), 256) : 0, b_rgb = out_rgb8 ? px * 3 : 0;
    if (b_lin + b_rgb) {
        if ((rc = ensure_stage(ctx, root, b_lin + b_rgb))) return rc;
        constexpr int NCH = 4;
        for (auto& e : root.ev_chunk)
            if (!e) RT_CUDA(ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        struct Part { char* dst; const char* src; char* stage; size_t bytes; };
        const Part parts[2] = {{(char*)out_linear_rgb, (const char*)root.d_mean, (char*)root.h_stage, out_linear_rgb ? px * 3 * sizeof(float) : 0},
                               {(char*)out_rgb8, (const char*)root.d_rgb8, (char*)root.h_stage + b_lin, b_rgb}};
        for (const Part& pt : parts) {
            if (!pt.bytes) continue;
            if (host_pinned(pt.dst)) {   // the caller's buffer is page-locked (rt_host_alloc / registered): the device writes it directly
                RT_CUDA(ctx, cudaMemcpyAsync(pt.dst, pt.src, pt.bytes, cudaMemcpyDeviceToHost, root.stream));
                continue;
            }
            const size_t step = align_up((pt.bytes + NCH - 1) / NCH, 4096);
            for (int c = 0; c < NCH; ++c) {
                const size_t off = std::min(pt.bytes, (size_t)c * step), len = std::min(pt.bytes - off, step);
                if (len) RT_CUDA(ctx, cudaMemcpyAsync(pt.stage + off, pt.src + off, len, cudaMemcpyDeviceToHost, root.stream));
                RT_CUDA(ctx, cudaEventRecord(root.ev_chunk[c], root.stream));
            }
            for (int c = 0; c < NCH; ++c) {
                const size_t off = std::min(pt.bytes, (size_t)c * step), len = std::min(pt.bytes - off, step);
                RT_CUDA(ctx, cudaEventSynchronize(root.ev_chunk[c]));
                if (len) memcpy(pt.dst + off, pt.stage + off, len);
            }
        }
    }
    RT_CUDA(ctx, cudaStreamSynchronize(root.stream));
    for (int g = 1; g < G; ++g) {
        RT_CUDA(ctx, cudaSetDevice(ctx->devs[g].dev));
        RT_CUDA(ctx, cudaStreamSynchronize(ctx->devs[g].stream));
    }
    cudaSetDevice(root.dev);
    if (G > 1) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, root.ev_r0, root.ev_r1) == cudaSuccess) ctx->reduce_ms += ms;
        cudaGetLastError();
    }
    return RT_OK;
}

int rt_host_alloc(rt_ctx* ctx, size_t bytes, void** out) {
    if (!out || bytes == 0) return ctx ? fail(ctx, RT_ERR_ARG, "rt_host_alloc: bad arguments") : RT_ERR_ARG;
    *out = nullptr;
    if (ctx && !ctx->devs.empty()) cudaSetDevice(ctx->devs[0].dev);
    const cudaError_t e = cudaHostAlloc(out, bytes, cudaHostAllocPortable);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(ctx, RT_ERR_CUDA, std::string("cudaHostAlloc: ") + cudaGetErrorString(e));
    }
    return RT_OK;
}

int rt_host_free(rt_ctx* ctx, void* p) {
    if (!p) return RT_OK;
    const cudaError_t e = cudaFreeHost(p);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(ctx, RT_ERR_CUDA, std::string("cudaFreeHost: ") + cudaGetErrorString(e));
    }
    return RT_OK;
}

int rt_trace_paths(rt_ctx* ctx, int nx, int ny, int n, const int32_t* pixel, const int32_t* sample, int max_depth, uint64_t seed,
                   int variant, float* out_radiance, int32_t* out_nrays, int32_t* out_term, int log_bounces, rt_path_bounce* out_log) {
    int rc = check_ready(ctx);
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if ((rc = check_camera_times(ctx))) return rc;
    if (nx <= 0 || ny <= 0 || n < 0 || max_depth < 0 || log_bounces < 0 || (n > 0 && (!pixel || !sample || !out_radiance || !out_nrays || !out_term)) ||
        (log_bounces > 0 && n > 0 && !out_log))
        return fail(ctx, RT_ERR_ARG, "bad trace_paths arguments");
    if ((long long)nx * ny > 0x7fffffffLL / 3) return fail(ctx, RT_ERR_ARG, "image too large");
    if (n == 0) return RT_OK;
    for (int q = 0; q < n; ++q)
        if (pixel[q] < 0 || pixel[q] >= nx * ny || sample[q] < 0 || sample[q] >= (1 << 24))
            return fail(ctx, RT_ERR_ARG, "pixel / sample index out of range");
    static_assert(sizeof(rt_path_bounce) == sizeof(PathBounce) && sizeof(PathBounce) == 40, "rt_path_bounce layout");
    DeviceBuffers& d = ctx->devs[0];
    RT_CUDA(ctx, cudaSetDevice(d.dev));
    const size_t b_i = align_up((size_t)n * 4, 256), b_f = align_up((size_t)n * 12, 256), b_l = align_up((size_t)n * log_bounces * sizeof(PathBounce), 256);
    char* buf = nullptr;   // its own allocation: the render below may grow the context's scratch
    RT_CUDA(ctx, cudaMalloc(&buf, 4 * b_i + b_f + b_l + 256));
    int* d_pix = (int*)buf;
    int* d_smp = (int*)(buf + b_i);
    int* d_nr = (int*)(buf + 2 * b_i);
    int* d_term = (int*)(buf + 3 * b_i);
    float* d_rad = (float*)(buf + 4 * b_i);
    PathBounce* d_log = log_bounces > 0 ? (PathBounce*)(buf + 4 * b_i + b_f) : nullptr;
    auto cleanup = [&](int code) { cudaStreamSynchronize(d.stream); cudaFree(buf); return code; };
    cudaError_t e;
    if ((e = cudaMemcpyAsync(d_pix, pixel, (size_t)n * 4, cudaMemcpyHostToDevice, d.stream)) != cudaSuccess ||
        (e = cudaMemcpyAsync(d_smp, sample, (size_t)n * 4, cudaMemcpyHostToDevice, d.stream)) != cudaSuccess ||
        (e = cudaMemsetAsync(d_nr, 0, 2 * b_i + b_f, d.stream)) != cudaSuccess ||
        (d_log && (e = cudaMemsetAsync(d_log, 0xff, (size_t)n * log_bounces * sizeof(PathBounce), d.stream)) != cudaSuccess))
        return cleanup(fail(ctx, RT_ERR_CUDA, std::string("trace_paths upload: ") + cudaGetErrorString(e)));
    RenderParams P{};
    P.nx = nx; P.ny = ny;
    P.sample_begin = 0; P.sample_count = 1;
    P.row_offset = 0; P.row_stride = 1; P.rows_in_shard = ny;
    P.max_depth = max_depth;
    P.key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
    P.sum = d_rad;
    P.total_work = (unsigned long long)n;
    P.path_pixel = d_pix; P.path_sample = d_smp; P.path_nrays = d_nr; P.path_term = d_term;
    P.path_log = d_log; P.path_log_n = log_bounces;
    if ((rc = launch_params(ctx, d, P, variant, d.stream))) return cleanup(rc);
    if ((e = cudaMemcpyAsync(out_radiance, d_rad, (size_t)n * 12, cudaMemcpyDeviceToHost, d.stream)) != cudaSuccess ||
        (e = cudaMemcpyAsync(out_nrays, d_nr, (size_t)n * 4, cudaMemcpyDeviceToHost, d.stream)) != cudaSuccess ||
        (e = cudaMemcpyAsync(out_term, d_term, (size_t)n * 4, cudaMemcpyDeviceToHost, d.stream)) != cudaSuccess ||
        (d_log && (e = cudaMemcpyAsync(out_log, d_log, (size_t)n * log_bounces * sizeof(PathBounce), cudaMemcpyDeviceToHost, d.stream)) != cudaSuccess) ||
        (e = cudaStreamSynchronize(d.stream)) != cudaSuccess)
        return cleanup(fail(ctx, RT_ERR_CUDA, std::string("trace_paths: ") + cudaGetErrorString(e)));
    // a logged slot that was never written (0xff fill) = the path had ended before that bounce
    if (out_log)
        for (size_t q = 0; q < (size_t)n * log_bounces; ++q)
            if (out_log[q].hit_id == -1 && std::isnan(out_log[q].t)) { memset(&out_log[q], 0, sizeof(rt_path_bounce)); out_log[q].hit_id = -2; }
    d.timed = false;
    return cleanup(RT_OK);
}

int rt_sample_device(rt_ctx* ctx, int kind, int n, uint64_t seed, float* out) {
    if (!ctx) return RT_ERR_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if ((kind != 0 && kind != 1) || n < 0 || (n > 0 && !out)) return fail(ctx, RT_ERR_ARG, "bad sample_device arguments");
    if (n == 0) return RT_OK;
    DeviceBuffers& d = ctx->devs[0];
    RT_CUDA(ctx, cudaSetDevice(d.dev));
    const int dim = kind == 0 ? 3 : 2;
    int rc;
    if ((rc = ensure_scratch(ctx, d, (size_t)n * dim * 4))) return rc;
    sampler_kernel<<<(n + 255) / 256, 256, 0, d.stream>>>(kind, n, make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)), (float*)d.scratch);
    RT_CUDA(ctx, cudaGetLastError());
    RT_CUDA(ctx, cudaMemcpyAsync(out, d.scratch, (size_t)n * dim * 4, cudaMemcpyDeviceToHost, d.stream));
    RT_CUDA(ctx, cudaStreamSynchronize(d.stream));
    return RT_OK;
}

int rt_trace_primary(rt_ctx* ctx, int n, const float* origins, const float* dirs, const float* times, double tmin,
                     double tmax, double* out_t, int32_t* out_id) {
    int rc = check_ready(ctx);
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (n < 0 || (n > 0 && (!origins || !dirs || !out_t || !out_id))) return fail(ctx, RT_ERR_ARG, "bad trace arguments");
    if (!(tmin >= 0.0)) return fail(ctx, RT_ERR_ARG, "tmin must be >= 0: the cull discards spheres behind the origin");
    if (n == 0) return RT_OK;
    {
        double lo = 0.0, hi = 0.0;
        if (times) {
            lo = INFINITY; hi = -INFINITY;
            for (int i = 0; i < n; ++i) { lo = std::min(lo, (double)times[i]); hi = std::max(hi, (double)times[i]); }
        }
        if ((rc = ensure_window(ctx, lo, hi))) return rc;
    }
    DeviceBuffers& d = ctx->devs[0];
    RT_CUDA(ctx, cudaSetDevice(d.dev));
    size_t b_o = align_up((size_t)n * 12, 256), b_t = align_up((size_t)n * 4, 256), b_ot = align_up((size_t)n * 8, 256);
    if ((rc = ensure_scratch(ctx, d, 2 * b_o + 2 * b_t + b_ot))) return rc;
    char* base = (char*)d.scratch;
    float* d_o = (float*)base;
    float* d_d = (float*)(base + b_o);
    float* d_tm = (float*)(base + 2 * b_o);
    int* d_id = (int*)(base + 2 * b_o + b_t);
    double* d_t = (double*)(base + 2 * b_o + 2 * b_t);
    RT_CUDA(ctx, cudaMemcpyAsync(d_o, origins, (size_t)n * 12, cudaMemcpyHostToDevice, d.stream));
    RT_CUDA(ctx, cudaMemcpyAsync(d_d, dirs, (size_t)n * 12, cudaMemcpyHostToDevice, d.stream));
    if (times) RT_CUDA(ctx, cudaMemcpyAsync(d_tm, times, (size_t)n * 4, cudaMemcpyHostToDevice, d.stream));
    if (ctx->accel == RT_ACCEL_BVH) {
        if ((rc = ensure_bvh(ctx))) return rc;
        TraceParamsB B{};
        B.sc = d.sc; B.n = n; B.origins = d_o; B.dirs = d_d; B.times = times ? d_tm : nullptr;
        B.tmin = tmin; B.tmax = tmax; B.out_t = d_t; B.out_id = d_id;
        B.stats = nullptr;
        if (ctx->generic) trace_bvh_kernel<true><<<(n + 127) / 128, 128, 0, d.stream>>>(B);
        else trace_bvh_kernel<false><<<(n + 127) / 128, 128, 0, d.stream>>>(B);
        RT_CUDA(ctx, cudaGetLastError());
        RT_CUDA(ctx, cudaMemcpyAsync(out_t, d_t, (size_t)n * 8, cudaMemcpyDeviceToHost, d.stream));
        RT_CUDA(ctx, cudaMemcpyAsync(out_id, d_id, (size_t)n * 4, cudaMemcpyDeviceToHost, d.stream));
        RT_CUDA(ctx, cudaStreamSynchronize(d.stream));
        return RT_OK;
    }
    TraceParams P{};
    P.sc = d.sc; P.n = n; P.origins = d_o; P.dirs = d_d; P.times = times ? d_tm : nullptr;
    P.tmin = tmin; P.tmax = tmax; P.out_t = d_t; P.out_id = d_id; P.cull_cap = ctx->cull_cap; P.preloaded = ctx->preloaded;
    void (*kern)(const TraceParams) = ctx->generic ? trace_kernel<kR, kBlock, true> : trace_kernel<kR, kBlock, false>;
    size_t smem = mega_smem_bytes(ctx->cull_cap);
    int bps = 0;
    if ((rc = configure_kernel(ctx, kern, smem, &bps))) return rc;
    int want = (int)(((long long)n + kBlock * kR - 1) / (kBlock * kR));
    int grid = std::max(1, std::min(d.sm_count * bps, want));
    kern<<<grid, kBlock, smem, d.stream>>>(P);
    RT_CUDA(ctx, cudaGetLastError());
    RT_CUDA(ctx, cudaMemcpyAsync(out_t, d_t, (size_t)n * 8, cudaMemcpyDeviceToHost, d.stream));
    RT_CUDA(ctx, cudaMemcpyAsync(out_id, d_id, (size_t)n * 4, cudaMemcpyDeviceToHost, d.stream));
    RT_CUDA(ctx, cudaStreamSynchronize(d.stream));
    return RT_OK;
}

int rt_cull_check(rt_ctx* ctx, int n, const float* origins, const float* dirs, const float* times, double tmin, double tmax,
                  uint64_t out[3]) {
    int rc = check_ready(ctx);
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (n < 0 || !out || (n > 0 && (!origins || !dirs))) return fail(ctx, RT_ERR_ARG, "bad cull_check arguments");
    if (!(tmin >= 0.0)) return fail(ctx, RT_ERR_ARG, "tmin must be >= 0: the cull discards spheres behind the origin");
    out[0] = out[1] = out[2] = 0;
    if (n == 0) return RT_OK;
    {
        double lo = 0.0, hi = 0.0;
        if (times) {
            lo = INFINITY; hi = -INFINITY;
            for (int i = 0; i < n; ++i) { lo = std::min(lo, (double)times[i]); hi = std::max(hi, (double)times[i]); }
        }
        if ((rc = ensure_window(ctx, lo, hi))) return rc;
    }
    DeviceBuffers& d = ctx->devs[0];
    RT_CUDA(ctx, cudaSetDevice(d.dev));
    size_t b_o = align_up((size_t)n * 12, 256), b_t = align_up((size_t)n * 4, 256);
    if ((rc = ensure_scratch(ctx, d, 2 * b_o + b_t + 256))) return rc;
    char* base = (char*)d.scratch;
    float* d_o = (float*)base;
    float* d_d = (float*)(base + b_o);
    float* d_tm = (float*)(base + 2 * b_o);
    unsigned long long* d_out = (unsigned long long*)(base + 2 * b_o + b_t);
    RT_CUDA(ctx, cudaMemcpyAsync(d_o, origins, (size_t)n * 12, cudaMemcpyHostToDevice, d.stream));
    RT_CUDA(ctx, cudaMemcpyAsync(d_d, dirs, (size_t)n * 12, cudaMemcpyHostToDevice, d.stream));
    if (times) RT_CUDA(ctx, cudaMemcpyAsync(d_tm, times, (size_t)n * 4, cudaMemcpyHostToDevice, d.stream));
    RT_CUDA(ctx, cudaMemsetAsync(d_out, 0, 3 * sizeof(unsigned long long), d.stream));
    if (ctx->opt.cull_tc && ctx->tc_tiles > 0) {   // (whatever the list length: this is the diagnostic)
        // option cull_tc: check the tensor-core cull by running the PRODUCTION kernel over a queue of these rays
        const size_t cap = align_up(std::max<size_t>((size_t)n, 1u << 18), 128);   // (room for the warps' 64-slot pair reservations of every pass)
        if ((rc = ensure_lane(ctx, d, 0, cap))) return rc;
        DeviceBuffers::WaveLane& L = d.lanes[0];
        L.best_clean = false;
        const int words = (ctx->n_cull + 31) / 32;
        unsigned* d_mask = nullptr;
        RT_CUDA(ctx, cudaMalloc(&d_mask, (size_t)n * words * sizeof(unsigned)));
        RT_CUDA(ctx, cudaMemsetAsync(d_mask, 0, (size_t)n * words * sizeof(unsigned), d.stream));
        WaveParams W{};
        W.base.sc = d.sc;
        W.base.cam = ctx->cam;
        W.base.counters = d.d_counters;
        W.base.work_counter = d.d_counters + DC_COUNT;
        W.base.max_depth = 1;
        W.queue[0] = L.queue;
        W.queue[1] = L.queue + 3 * L.entries;
        W.best_t = L.best;
        W.best_key = L.best + L.entries;
        W.pairs = L.pairs;
        W.cands = L.cands;
        W.cand_t = L.cand_t;
        W.cand_count = L.cand_count;
        W.st = L.state;
        W.capacity = (int)L.entries;
        W.pair_cap = (unsigned)std::min<size_t>(L.entries * kPairsPerEntry, 0xfffffff0u);
        wf_fill_best<<<d.sm_count * 4, 256, 0, d.stream>>>(L.best, L.best + L.entries, L.entries);
#ifdef RT_TC_CHECK
        RT_CUDA(ctx, cudaMemsetAsync(L.pairs, 0xDD, (size_t)W.pair_cap * sizeof(uint2), d.stream));
#endif
        tc_check_fill<<<(n + 127) / 128, 128, 0, d.stream>>>(W, n, d_o, d_d, times ? d_tm : nullptr);
        const int launch_tiles = std::min(ctx->tc_tiles, (int)tc::MAX_TILES);
        W.tc_slots = tc::slots_for(launch_tiles, 227 * 1024);
        const size_t tc_smem = tc::smem_bytes(launch_tiles, W.tc_slots);
        RT_CUDA(ctx, cudaFuncSetAttribute(wf_cull_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc_smem));
        for (int t0 = 0, pass = 0; t0 < ctx->tc_tiles; t0 += tc::MAX_TILES, ++pass) {
            W.tc_tile0 = t0;
            W.tc_launch_tiles = std::min((int)tc::MAX_TILES, ctx->tc_tiles - t0);
            W.tc_pass = pass;
            wf_cull_tc<<<d.sm_count, tc::THREADS, tc_smem, d.stream>>>(W);
        }
        tc_check_mark<<<d.sm_count * 4, 256, 0, d.stream>>>(W, d_mask, words);
        tc_check_compare<<<(n + 127) / 128, 128, 0, d.stream>>>(W, n, tmin, tmax, d_mask, words, d_out);
        cudaError_t e = cudaStreamSynchronize(d.stream);
        cudaFree(d_mask);
        if (e != cudaSuccess) return fail(ctx, RT_ERR_CUDA, std::string("tensor-core cull check: ") + cudaGetErrorString(e));
    } else {
        cull_check_kernel<<<(n + 127) / 128, 128, 0, d.stream>>>(d.sc, n, d_o, d_d, times ? d_tm : nullptr, tmin, tmax, d_out);
    }
    RT_CUDA(ctx, cudaGetLastError());
    unsigned long long h[3];
    RT_CUDA(ctx, cudaMemcpyAsync(h, d_out, sizeof(h), cudaMemcpyDeviceToHost, d.stream));
    RT_CUDA(ctx, cudaStreamSynchronize(d.stream));
    for (int i = 0; i < 3; ++i) out[i] = h[i];
    return RT_OK;
}

int rt_generate_rays(rt_ctx* ctx, int n, int nx, int ny, const int32_t* ij, const int32_t* s, uint64_t seed,
                     float* out_origin, float* out_dir, float* out_time, float* out_rand) {
    if (!ctx) return RT_ERR_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (!ctx->has_cam) return fail(ctx, RT_ERR_STATE, "rt_set_camera has not been called");
    if (n < 0 || nx <= 0 || ny <= 0 || (n > 0 && (!ij || !s || !out_origin || !out_dir || !out_time)))
        return fail(ctx, RT_ERR_ARG, "bad generate_rays arguments");
    if (n == 0) return RT_OK;
    DeviceBuffers& d = ctx->devs[0];
    RT_CUDA(ctx, cudaSetDevice(d.dev));
    size_t b_ij = align_up((size_t)n * 8, 256), b_s = align_up((size_t)n * 4, 256), b_v = align_up((size_t)n * 12, 256),
           b_r = align_up((size_t)n * 20, 256);
    int rc;
    if ((rc = ensure_scratch(ctx, d, b_ij + 2 * b_s + 2 * b_v + b_r))) return rc;
    char* base = (char*)d.scratch;
    int* d_ij = (int*)base;
    int* d_s = (int*)(base + b_ij);
    float* d_o = (float*)(base + b_ij + b_s);
    float* d_d = (float*)(base + b_ij + b_s + b_v);
    float* d_t = (float*)(base + b_ij + b_s + 2 * b_v);
    float* d_r = (float*)(base + b_ij + 2 * b_s + 2 * b_v);
    RT_CUDA(ctx, cudaMemcpyAsync(d_ij, ij, (size_t)n * 8, cudaMemcpyHostToDevice, d.stream));
    RT_CUDA(ctx, cudaMemcpyAsync(d_s, s, (size_t)n * 4, cudaMemcpyHostToDevice, d.stream));
    genrays_kernel<<<(n + 255) / 256, 256, 0, d.stream>>>(ctx->cam, n, nx, ny, d_ij, d_s,
                                                         make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)), d_o, d_d, d_t,
                                                         out_rand ? d_r : nullptr);
    RT_CUDA(ctx, cudaGetLastError());
    RT_CUDA(ctx, cudaMemcpyAsync(out_origin, d_o, (size_t)n * 12, cudaMemcpyDeviceToHost, d.stream));
    RT_CUDA(ctx, cudaMemcpyAsync(out_dir, d_d, (size_t)n * 12, cudaMemcpyDeviceToHost, d.stream));
    RT_CUDA(ctx, cudaMemcpyAsync(out_time, d_t, (size_t)n * 4, cudaMemcpyDeviceToHost, d.stream));
    if (out_rand) RT_CUDA(ctx, cudaMemcpyAsync(out_rand, d_r, (size_t)n * 20, cudaMemcpyDeviceToHost, d.stream));
    RT_CUDA(ctx, cudaStreamSynchronize(d.stream));
    return RT_OK;
}

int rt_shade_batch(rt_ctx* ctx, int n, const float* origins, const float* dirs, const float* times, const int32_t* hit_id,
                   const double* hit_t, const float* ball, const float* u01v, float* out_origin, float* out_dir,
                   float* out_atten, float* out_emitted, int32_t* out_flags) {
    int rc = check_ready(ctx);
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (n < 0 || (n > 0 && (!origins || !dirs || !hit_id || !hit_t || !ball || !u01v || !out_origin || !out_dir ||
                            !out_atten || !out_emitted || !out_flags)))
        return fail(ctx, RT_ERR_ARG, "bad shade_batch arguments");
    if (n == 0) return RT_OK;
    DeviceBuffers& d = ctx->devs[0];
    RT_CUDA(ctx, cudaSetDevice(d.dev));
    size_t b3 = align_up((size_t)n * 12, 256), b1 = align_up((size_t)n * 4, 256), b8 = align_up((size_t)n * 8, 256);
    if ((rc = ensure_scratch(ctx, d, 7 * b3 + 4 * b1 + b8))) return rc;
    char* p = (char*)d.scratch;
    float* d_o = (float*)p; p += b3;
    float* d_d = (float*)p; p += b3;
    float* d_ball = (float*)p; p += b3;
    float* d_oo = (float*)p; p += b3;
    float* d_od = (float*)p; p += b3;
    float* d_oa = (float*)p; p += b3;
    float* d_oe = (float*)p; p += b3;
    float* d_tm = (float*)p; p += b1;
    float* d_u = (float*)p; p += b1;
    int* d_id = (int*)p; p += b1;
    int* d_fl = (int*)p; p += b1;
    double* d_ht = (double*)p;
    RT_CUDA(ctx, cudaMemcpyAsync(d_o, origins, (size_t)n * 12, cudaMemcpyHostToDevice, d.stream));
    RT_CUDA(ctx, cudaMemcpyAsync(d_d, dirs, (size_t)n * 12, cudaMemcpyHostToDevice, d.stream));
    RT_CUDA(ctx, cudaMemcpyAsync(d_ball, ball, (size_t)n * 12, cudaMemcpyHostToDevice, d.stream));
    if (times) RT_CUDA(ctx, cudaMemcpyAsync(d_tm, times, (size_t)n * 4, cudaMemcpyHostToDevice, d.stream));
    RT_CUDA(ctx, cudaMemcpyAsync(d_u, u01v, (size_t)n * 4, cudaMemcpyHostToDevice, d.stream));
    RT_CUDA(ctx, cudaMemcpyAsync(d_id, hit_id, (size_t)n * 4, cudaMemcpyHostToDevice, d.stream));
    RT_CUDA(ctx, cudaMemcpyAsync(d_ht, hit_t, (size_t)n * 8, cudaMemcpyHostToDevice, d.stream));
    shade_kernel<<<(n + 255) / 256, 256, 0, d.stream>>>(d.sc, n, d_o, d_d, times ? d_tm : nullptr, d_id, d_ht, d_ball, d_u,
                                                       d_oo, d_od, d_oa, d_oe, d_fl);
    RT_CUDA(ctx, cudaGetLastError());
    RT_CUDA(ctx, cudaMemcpyAsync(out_origin, d_oo, (size_t)n * 12, cudaMemcpyDeviceToHost, d.stream));
    RT_CUDA(ctx, cudaMemcpyAsync(out_dir, d_od, (size_t)n * 12, cudaMemcpyDeviceToHost, d.stream));
    RT_CUDA(ctx, cudaMemcpyAsync(out_atten, d_oa, (size_t)n * 12, cudaMemcpyDeviceToHost, d.stream));
    RT_CUDA(ctx, cudaMemcpyAsync(out_emitted, d_oe, (size_t)n * 12, cudaMemcpyDeviceToHost, d.stream));
    RT_CUDA(ctx, cudaMemcpyAsync(out_flags, d_fl, (size_t)n * 4, cudaMemcpyDeviceToHost, d.stream));
    RT_CUDA(ctx, cudaStreamSynchronize(d.stream));
    return RT_OK;
}

int rt_measure_fp32_peak(rt_ctx* ctx, double* out_ffma_tflops, double* out_ffma2_tflops) {
    if (!ctx) return RT_ERR_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    DeviceBuffers& d = ctx->devs[0];
    RT_CUDA(ctx, cudaSetDevice(d.dev));
    const int blocks = d.sm_count * 8, threads = 256, iters = 1 << 15;
    int rc;
    if ((rc = ensure_scratch(ctx, d, (size_t)blocks * threads * 4))) return rc;
    float* out = (float*)d.scratch;
    double best[2] = {0, 0};
    for (int variant = 0; variant < 2; ++variant) {
        for (int rep = 0; rep < 4; ++rep) {
            RT_CUDA(ctx, cudaEventRecord(d.ev0, d.stream));
            if (variant == 0) ffma_peak_kernel<false><<<blocks, threads, 0, d.stream>>>(out, iters, 1.0000001f, 1e-7f);
            else ffma_peak_kernel<true><<<blocks, threads, 0, d.stream>>>(out, iters, 1.0000001f, 1e-7f);
            RT_CUDA(ctx, cudaGetLastError());
            RT_CUDA(ctx, cudaEventRecord(d.ev1, d.stream));
            RT_CUDA(ctx, cudaEventSynchronize(d.ev1));
            float ms = 0;
            RT_CUDA(ctx, cudaEventElapsedTime(&ms, d.ev0, d.ev1));
            double flops = 2.0 * 16.0 * (double)iters * (double)blocks * threads;   // 16 FMA per thread per iter either way
            if (rep > 0) best[variant] = std::max(best[variant], flops / (ms * 1e-3) / 1e12);
        }
    }
    if (out_ffma_tflops) *out_ffma_tflops = best[0];
    if (out_ffma2_tflops) *out_ffma2_tflops = best[1];
    d.timed = false;
    return RT_OK;
}

int rt_get_counters(rt_ctx* ctx, uint64_t out[RT_CTR_COUNT]) {
    if (!ctx || !out) return RT_ERR_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    unsigned long long dc[DC_COUNT];
    uint64_t total[DC_COUNT] = {0};
    float max_ms = 0.f;
    for (auto& d : ctx->devs) {
        RT_CUDA(ctx, cudaSetDevice(d.dev));
        RT_CUDA(ctx, cudaDeviceSynchronize());
        RT_CUDA(ctx, cudaMemcpy(dc, d.d_counters, sizeof(dc), cudaMemcpyDeviceToHost));
        for (int i = 0; i < DC_COUNT; ++i) total[i] += dc[i];
        if (!d.trace_meta.empty() && d.d_trace && getenv("RT_TRACE")) {   // timeline of the last traced render
            std::vector<TraceRec> rec(d.trace_meta.size());
            RT_CUDA(ctx, cudaMemcpy(rec.data(), d.d_trace, rec.size() * sizeof(TraceRec), cudaMemcpyDeviceToHost));
            unsigned long long t0 = ~0ull;
            for (auto& r : rec) if (r.t_end) t0 = std::min(t0, r.t_start);
            if (FILE* f = fopen(getenv("RT_TRACE"), "a")) {   // appended: one block per traced render that was followed by rt_get_counters
                fprintf(f, "# device %d, %zu launches: kernel lane iteration start_us end_us duration_us (%%globaltimer, relative to the first kernel)\n", d.dev, rec.size());
                for (size_t i = 0; i < rec.size(); ++i) {
                    if (!rec[i].t_end) continue;   // the launch found an empty queue
                    fprintf(f, "%-9s %d %3d %10.1f %10.1f %9.1f\n", d.trace_meta[i].kernel, d.trace_meta[i].lane, d.trace_meta[i].iter,
                            (rec[i].t_start - t0) * 1e-3, (rec[i].t_end - t0) * 1e-3, (rec[i].t_end - rec[i].t_start) * 1e-3);
                }
                fclose(f);
            }
            d.trace_meta.clear();
        }
        if (d.timed) {
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, d.ev0, d.ev1) == cudaSuccess) d.last_ms = ms;
            cudaGetLastError();
        }
        max_ms = std::max(max_ms, d.last_ms);
    }
    cudaSetDevice(ctx->devs[0].dev);
    memset(out, 0, sizeof(uint64_t) * RT_CTR_COUNT);
    out[RT_CTR_RAYS] = total[DC_RAYS];
    out[RT_CTR_SPHERE_TESTS] = total[DC_RAYS] * (uint64_t)ctx->n_spheres;
    out[RT_CTR_SAMPLES] = total[DC_SAMPLES];
    out[RT_CTR_TERM_LIGHT] = total[DC_TERM_LIGHT];
    out[RT_CTR_TERM_ABSORB] = total[DC_TERM_ABSORB];
    out[RT_CTR_TERM_DEPTH] = total[DC_TERM_DEPTH];
    out[RT_CTR_TERM_MISS] = total[DC_TERM_MISS];
    out[RT_CTR_KERNEL_NS] = (uint64_t)((double)max_ms * 1e6);
    out[RT_CTR_CANDIDATES] = total[DC_CANDIDATES];
    out[RT_CTR_DIRECT_TESTS] = total[DC_DIRECT];
    out[RT_CTR_BVH_NODE_TESTS] = total[DC_BVH_NODES];
    if (ctx->accel == RT_ACCEL_BVH) out[RT_CTR_SPHERE_TESTS] = total[DC_CANDIDATES] + total[DC_DIRECT];   // exact tests actually made
    out[RT_CTR_KERNEL_LAUNCHES] = ctx->n_launches.load();
    out[RT_CTR_CULL_NS] = (uint64_t)(ctx->stage_ms[0] * 1e6);
    out[RT_CTR_REFINE_NS] = (uint64_t)(ctx->stage_ms[1] * 1e6);
    out[RT_CTR_TIEBREAK_NS] = (uint64_t)(ctx->stage_ms[2] * 1e6);
    out[RT_CTR_SHADE_NS] = (uint64_t)(ctx->stage_ms[3] * 1e6);
    out[RT_CTR_REDUCE_NS] = (uint64_t)(ctx->reduce_ms * 1e6);
    return RT_OK;
}

int rt_reset_counters(rt_ctx* ctx) {
    if (!ctx) return RT_ERR_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    for (auto& d : ctx->devs) {
        RT_CUDA(ctx, cudaSetDevice(d.dev));
        RT_CUDA(ctx, cudaDeviceSynchronize());
        RT_CUDA(ctx, cudaMemset(d.d_counters, 0, (DC_COUNT + 1) * sizeof(unsigned long long)));
    }
    cudaSetDevice(ctx->devs[0].dev);
    ctx->n_launches = 0;
    for (double& x : ctx->stage_ms) x = 0.0;
    ctx->reduce_ms = 0.0;
    return RT_OK;
}

int rt_set_profile(rt_ctx* ctx, int on) {
    if (!ctx) return RT_ERR_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->profile = on != 0;
    return RT_OK;
}

}  // extern "C"
