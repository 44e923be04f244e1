// bgx_api.cu — sections 2..6 of include/bgx.h: the engine handle and the batched GPU
// entry points.  Everything here launches the kernels of bgx_kernels.cuh / bgx_td.cuh on
// the engine's stream; there is no CPU path — without a device bgx_create fails.
#include "../../include/bgx.h"
#include "bgx_internal.h"
#include "bgx_kernels.cuh"
#include "bgx_td.cuh"
#include "bgx_twoply.cuh"
#include "bgx_rollout.cuh"

#include <dlfcn.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

using namespace bgx;

// an asynchronous lane of the batched make_move path: its own stream, work-queue counter,
// sharing buffer and staging buffers, so that two batches can be in flight at once
struct bgx_lane {
    cudaStream_t stream = nullptr;
    cudaEvent_t done = nullptr;
    unsigned long long *counter = nullptr;   // [0] work queue, [8..15] the 16 bucket totals of k_select_order
    StealResult *steal = nullptr;
    void *buf[11] = {};                      // [7] [10]: sorted queues (two slots), [8] [9]: ply and game id of bgx_play_ply_host_async
    size_t cap[11] = {};
    int order_slot = 0;                      // slot holding the queue the previous bgx_play_ply_host_async produced for its successor ...
    int64_t order_n = -1;                    // ... valid for a batch of exactly this many queries (-1: none)
    bool busy = false;
};
constexpr int kLanes = BGX_ASYNC_LANES;
constexpr size_t kCounterBytes = 256;        // work-queue counter; 16 x uint32 bucket totals at byte 64 (slot 0) and 128 (slot 1)

struct bgx_engine {
    int device = 0;
    cudaStream_t stream = nullptr;
    int sm_count = 0, clock_khz = 0;
    size_t global_mem = 0;
    // model
    float *flat = nullptr;        // [25604] state_dict order
    float *wt = nullptr;          // [198][128] W1 transposed (TD kernel)
    int32_t *fixed = nullptr;     // [198][128] W1 transposed in fixed point (ply kernels, k_evaluate)
    float *aux = nullptr;         // [4] derived scalars: [0] fixed-point scale S, [1] 1/S
    bool have_weights = false;
    // scratch ([12..31] belong to the two-ply path, [32..] to rollouts)
    static constexpr int kScratch = 40;
    void *dbuf[kScratch] = {};
    size_t dcap[kScratch] = {};
    unsigned long long *counter = nullptr;   // work queue
    unsigned long long *stats = nullptr;     // 8 counters
    double *dstats = nullptr;                // TD: sum of squared errors
    StealResult *steal = nullptr;            // [CTA][warp][16] sub-tree results of shared doubles (bgx_ply.cuh)
    int4 *zstash = nullptr;                  // [CTA][32 warps][32 lanes] pre-activation of a self-play warp's best afterstate (bgx_ply.cuh)
    uint32_t *uniq_tables = nullptr;
    uint32_t *uniq_gens = nullptr;           // per-warp generation of the exact-dedup tables
    int uniq_grid = 0;
    // self-play population
    long long n_slots = 0, first_id = 0, id_stride = 0;
    uint32_t seed_lo = 0, seed_hi = 0;
    int first_mover = 0, traj_cap = 0;
    bool record_chosen = false;
    int8_t *slots = nullptr, *traj_pre = nullptr, *traj_chosen = nullptr;
    int32_t *ply = nullptr;
    long long *game_id = nullptr;
    // TD
    float *td_partial = nullptr;             // [td_grid][25604] per-CTA delta accumulators
    float *td_delta = nullptr;               // [25604] summed delta of bgx_td_round_host
    float *td_home = nullptr;                // [td_grid][2][198][128] per-CTA home copies of W1 and its traces (k_td_replay)
    double *td_sched = nullptr;              // [2][64] lr / lambda by schedule index (bgx_td_replay_scheduled)
    unsigned long long *td_prof = nullptr;   // [16] phase cycles of the profiling variant of k_td_replay
    bool td_profile = false;
    int td_grid = 0;
    int lane_grid = -1;                      // CTAs of a k_select launch on an asynchronous lane: half the SMs, so that two lanes'
                                             // batches are resident at once (0: one per SM); this and the next: bgx_set_option
    long long select_order_max = 1 << 21;    // launches up to this many queries get a sorted queue (64 B of scratch per query)
    int select_urgent_min = 7, select_giant_min = kGiantMinChildren, select_urgent_from_pct = 0;   // k_select help policy
    int selfplay_warps = 20, select_warps = 20;   // warps per CTA of k_selfplay / k_select (measured best: 96 registers, 86 cache sets per warp)
    long long twoply_chunk = 0;              // replies per k_select launch of a two-ply call (0: kTwoplyChunk)
    bool twoply_timing = false;              // time the stages of a two-ply call (synchronises between them)
    double twoply_ms[4] = {};                // candidates, expand, replies, reduce: accumulated stage times
    long long rollout_chunk = 0;             // trials (games) per k_rollout launch, whole positions (0: kRolloutChunk)
    int rollout_warps = 20;                  // warps per CTA of k_rollout
    cudaEvent_t tp0 = nullptr, tp1 = nullptr;
    // bookkeeping
    long long launches = 0;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_sync = nullptr;
    bool timed = false;
    bgx_lane lanes[kLanes];
};

#define CU(call)                                                                              \
    do {                                                                                      \
        cudaError_t err__ = (call);                                                           \
        if (err__ != cudaSuccess) {                                                           \
            set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(err__)); \
            return BGX_E_CUDA;                                                                \
        }                                                                                     \
    } while (0)

#define NEED(cond, msg)                                   \
    do {                                                  \
        if (!(cond)) { set_error("%s: %s", __func__, msg); return BGX_E_INVALID; } \
    } while (0)

static int use(bgx_engine *e)
{
    if (!e) { set_error("null engine"); return BGX_E_INVALID; }
    CU(cudaSetDevice(e->device));
    return BGX_OK;
}
#define USE(e)                       \
    do {                             \
        int rc__ = use(e);           \
        if (rc__ != BGX_OK) return rc__; \
    } while (0)

static int scratch(bgx_engine *e, int i, size_t bytes, void **out)
{
    if (e->dcap[i] < bytes) {
        if (e->dbuf[i]) CU(cudaFree(e->dbuf[i]));
        e->dbuf[i] = nullptr;
        e->dcap[i] = 0;
        size_t want = bytes + bytes / 4 + 256;
        CU(cudaMalloc(&e->dbuf[i], want));
        e->dcap[i] = want;
    }
    *out = e->dbuf[i];
    return BGX_OK;
}

static int tick_(bgx_engine *e) { CU(cudaEventRecord(e->ev0, e->stream)); return BGX_OK; }
static int tock_(bgx_engine *e) { CU(cudaEventRecord(e->ev1, e->stream)); e->timed = true; return BGX_OK; }
#define tick(e) do { const int rc__ = tick_(e); if (rc__ != BGX_OK) return rc__; } while (0)
#define tock(e) do { const int rc__ = tock_(e); if (rc__ != BGX_OK) return rc__; } while (0)

static int game_grid(bgx_engine *e) { return e->sm_count; }   // persistent: one 16-warp CTA per SM

extern "C" {

int bgx_device_count(int *n)
{
    if (!n) { set_error("bgx_device_count: null"); return BGX_E_INVALID; }
    int c = 0;
    cudaError_t err = cudaGetDeviceCount(&c);
    if (err != cudaSuccess) { *n = 0; set_error("cudaGetDeviceCount: %s", cudaGetErrorString(err)); return BGX_E_NO_DEVICE; }
    *n = c;
    return BGX_OK;
}

// everything bgx_create allocates hangs off *e, so a failure half-way is undone by bgx_destroy
static int create_into(bgx_engine *e, int device, const cudaDeviceProp &prop)
{
    e->device = device;
    e->sm_count = prop.multiProcessorCount;
    e->global_mem = prop.totalGlobalMem;
    CU(cudaDeviceGetAttribute(&e->clock_khz, cudaDevAttrClockRate, device));
    CU(cudaMalloc(&e->flat, BGX_NPARAMS_PADDED * sizeof(float)));
    CU(cudaMemset(e->flat, 0, BGX_NPARAMS_PADDED * sizeof(float)));
    CU(cudaMalloc(&e->wt, kTableBytes));
    CU(cudaMalloc(&e->fixed, kFixedBytes));
    CU(cudaMalloc(&e->aux, 4 * sizeof(float)));
    CU(cudaMemset(e->aux, 0, 4 * sizeof(float)));
    CU(cudaMalloc(&e->counter, kCounterBytes));
    CU(cudaMalloc(&e->stats, 16 * sizeof(unsigned long long)));
    CU(cudaMalloc(&e->dstats, 2 * sizeof(double)));
    CU(cudaMalloc(&e->steal, (size_t)e->sm_count * 32 * kStealMaxResults * sizeof(StealResult)));
    CU(cudaMalloc(&e->zstash, (size_t)e->sm_count * 32 * 32 * sizeof(int4)));
    CU(cudaEventCreate(&e->ev0));
    CU(cudaEventCreate(&e->ev1));
    CU(cudaEventCreateWithFlags(&e->ev_sync, cudaEventDisableTiming));
    CU(cudaFuncSetAttribute(k_evaluate, cudaFuncAttributeMaxDynamicSharedMemorySize, kEvalSmem));
    CU(cudaFuncSetAttribute(k_encode, cudaFuncAttributeMaxDynamicSharedMemorySize, kEncSmem));
    CU(cudaFuncSetAttribute(k_candidates, cudaFuncAttributeMaxDynamicSharedMemorySize, kEvalSmem));
    CU(cudaFuncSetAttribute(k_twoply_reduce, cudaFuncAttributeMaxDynamicSharedMemorySize, kEvalSmem));
    e->lane_grid = e->sm_count / 2;
    static_assert(ply_smem<16, 109>() <= 232448 && ply_smem<20, 86>() <= 232448 && ply_smem<24, 72>() <= 232448 && ply_smem<32, 53>() <= 232448,
                  "fused ply kernels: shared memory per CTA");
#define BGX_SMEM_ATTR(W, S)                                                                                                    \
    CU(cudaFuncSetAttribute(k_select<W, S, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, ply_smem<W, S>()));            \
    CU(cudaFuncSetAttribute(k_select<W, S, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, ply_smem<W, S>()));             \
    CU(cudaFuncSetAttribute(k_selfplay<W, S, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, ply_smem<W, S>()));          \
    CU(cudaFuncSetAttribute(k_selfplay<W, S, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, ply_smem<W, S>()));          \
    CU(cudaFuncSetAttribute(k_rollout<W, S>, cudaFuncAttributeMaxDynamicSharedMemorySize, ply_smem<W, S>()));
    BGX_SMEM_ATTR(16, 109)
    BGX_SMEM_ATTR(20, 86)
    BGX_SMEM_ATTR(24, 72)
    BGX_SMEM_ATTR(32, 53)
#undef BGX_SMEM_ATTR
    CU(cudaFuncSetAttribute(k_td_replay<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTdSmem));
    CU(cudaFuncSetAttribute(k_td_replay<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTdSmem));
    // the smallest carve-out that holds kTdCtasPerSm games (percent of the SM's 228 KB): the rest of the array is their L1
    CU(cudaFuncSetAttribute(k_td_replay<false>, cudaFuncAttributePreferredSharedMemoryCarveout, kTdCarveoutBytes * 100 / (228 * 1024)));
    CU(cudaFuncSetAttribute(k_td_replay<true>, cudaFuncAttributePreferredSharedMemoryCarveout, kTdCarveoutBytes * 100 / (228 * 1024)));
    return BGX_OK;
}

int bgx_create(int device, bgx_engine **out)
{
    if (!out) { set_error("bgx_create: null out"); return BGX_E_INVALID; }
    *out = nullptr;
    int n = 0;
    cudaError_t err = cudaGetDeviceCount(&n);
    if (err != cudaSuccess || n == 0) {
        set_error("bgx_create: no CUDA device (%s); libbgx has no CPU path", err == cudaSuccess ? "0 devices" : cudaGetErrorString(err));
        return BGX_E_NO_DEVICE;
    }
    if (device < 0 || device >= n) { set_error("bgx_create: device %d of %d", device, n); return BGX_E_INVALID; }
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) { set_error("bgx_create: device %d is sm_%d%d; libbgx is built for sm_100a only", device, prop.major, prop.minor); return BGX_E_NO_DEVICE; }
    bgx_engine *e = new bgx_engine();
    const int rc = create_into(e, device, prop);
    if (rc != BGX_OK) {                              // the message of the failing call survives the clean-up
        bgx_destroy(e);
        return rc;
    }
    *out = e;
    return BGX_OK;
}

// Tuning knobs of the fused ply kernels, for benchmarks and probes (the defaults are the measured best):
//   "selfplay_warps" / "select_warps"  warps per CTA of k_selfplay / k_select: 16, 20, 24 or 32
//   "select_lane_grid"                 CTAs of a launch on an asynchronous lane (0: one per SM; default: half the SMs)
//   "select_order_max"                 largest batch that gets a sorted queue
//   "select_urgent_min" / "select_giant_min" / "select_urgent_from_pct"   when a CTA helps a published double
//   "rollout_warps"                    warps per CTA of k_rollout: 16, 20, 24 or 32
//   "rollout_chunk"                    trials (games) per k_rollout launch, rounded down to whole positions (0: 2^24)
int bgx_set_option(bgx_engine *e, const char *key, int64_t value)
{
    if (!e || !key) { set_error("bgx_set_option: null"); return BGX_E_INVALID; }
    const std::string k(key);
    if (k == "selfplay_warps" || k == "select_warps" || k == "rollout_warps") {
        if (value != 16 && value != 20 && value != 24 && value != 32) { set_error("bgx_set_option: %s must be 16, 20, 24 or 32", key); return BGX_E_INVALID; }
        (k == "selfplay_warps" ? e->selfplay_warps : k == "select_warps" ? e->select_warps : e->rollout_warps) = (int)value;
    } else if (k == "select_lane_grid") {
        if (value < 0 || value > e->sm_count) { set_error("bgx_set_option: select_lane_grid is 0 .. %d", e->sm_count); return BGX_E_INVALID; }
        e->lane_grid = (int)value;
    } else if (k == "select_order_max") e->select_order_max = (long long)value;
    else if (k == "select_urgent_min") e->select_urgent_min = (int)value;
    else if (k == "select_giant_min") e->select_giant_min = (int)value;
    else if (k == "select_urgent_from_pct") e->select_urgent_from_pct = (int)value;
    else if (k == "twoply_chunk") {
        if (value < 0) { set_error("bgx_set_option: twoply_chunk must be >= 0"); return BGX_E_INVALID; }
        e->twoply_chunk = (long long)value;
    } else if (k == "twoply_timing") e->twoply_timing = value != 0;
    else if (k == "rollout_chunk") {
        if (value < 0) { set_error("bgx_set_option: rollout_chunk must be >= 0"); return BGX_E_INVALID; }
        e->rollout_chunk = (long long)value;
    }
    else { set_error("bgx_set_option: unknown option '%s'", key); return BGX_E_INVALID; }
    return BGX_OK;
}

int bgx_destroy(bgx_engine *e)
{
    if (!e) return BGX_OK;
    cudaSetDevice(e->device);
    cudaDeviceSynchronize();
    for (int i = 0; i < bgx_engine::kScratch; i++) cudaFree(e->dbuf[i]);
    cudaFree(e->flat); cudaFree(e->wt); cudaFree(e->fixed); cudaFree(e->aux); cudaFree(e->counter); cudaFree(e->stats); cudaFree(e->dstats); cudaFree(e->steal); cudaFree(e->zstash);
    cudaFree(e->uniq_tables); cudaFree(e->uniq_gens); cudaFree(e->slots); cudaFree(e->traj_pre); cudaFree(e->traj_chosen);
    cudaFree(e->ply); cudaFree(e->game_id); cudaFree(e->td_partial); cudaFree(e->td_delta); cudaFree(e->td_prof); cudaFree(e->td_home); cudaFree(e->td_sched);
    if (e->ev0) cudaEventDestroy(e->ev0);
    if (e->ev1) cudaEventDestroy(e->ev1);
    if (e->ev_sync) cudaEventDestroy(e->ev_sync);
    if (e->tp0) cudaEventDestroy(e->tp0);
    if (e->tp1) cudaEventDestroy(e->tp1);
    for (bgx_lane &l : e->lanes) {
        if (l.stream) cudaStreamDestroy(l.stream);
        if (l.done) cudaEventDestroy(l.done);
        cudaFree(l.counter); cudaFree(l.steal);
        for (void *b : l.buf) cudaFree(b);
    }
    delete e;
    return BGX_OK;
}

int bgx_set_stream(bgx_engine *e, void *cuda_stream)
{
    USE(e);
    e->stream = (cudaStream_t)cuda_stream;
    return BGX_OK;
}

int bgx_synchronize(bgx_engine *e)
{
    USE(e);
    CU(cudaStreamSynchronize(e->stream));
    return BGX_OK;
}

// weights may not change under a batch in flight: a lane's k_select reads the tables on its own stream
static int lanes_idle(bgx_engine *e, const char *who)
{
    for (int i = 0; i < kLanes; i++)
        if (e->lanes[i].busy) { set_error("%s: lane %d has a batch in flight (bgx_lane_wait first)", who, i); return BGX_E_STATE; }
    return BGX_OK;
}

static int rebuild_table(bgx_engine *e)
{
    k_build_table<<<(kTableFloats + 255) / 256, 256, 0, e->stream>>>(e->flat, e->wt);
    k_fixed_scale<<<1, kHidden, 0, e->stream>>>(e->flat, e->aux);
    k_build_fixed<<<(kFixedInts + 255) / 256, 256, 0, e->stream>>>(e->flat, e->aux, e->fixed);
    e->launches += 3;
    CU(cudaGetLastError());
    return BGX_OK;
}

int bgx_set_weights(bgx_engine *e, const float *W1, const float *b1, const float *w2, const float *b2)
{
    USE(e);
    NEED(W1 && b1 && w2 && b2, "null weight pointer");
    if (int rc = lanes_idle(e, "bgx_set_weights")) return rc;
    std::vector<float> flat(BGX_NPARAMS_PADDED, 0.f);
    std::memcpy(flat.data(), W1, kTableFloats * sizeof(float));
    std::memcpy(flat.data() + kTableFloats, b1, kHidden * sizeof(float));
    std::memcpy(flat.data() + kTableFloats + kHidden, w2, kHidden * sizeof(float));
    flat[kTableFloats + 2 * kHidden] = b2[0];
    CU(cudaMemcpyAsync(e->flat, flat.data(), flat.size() * sizeof(float), cudaMemcpyHostToDevice, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    e->have_weights = true;
    return rebuild_table(e);
}

int bgx_get_weights(bgx_engine *e, float *W1, float *b1, float *w2, float *b2)
{
    USE(e);
    NEED(W1 && b1 && w2 && b2, "null weight pointer");
    std::vector<float> flat(BGX_NPARAMS_PADDED);
    CU(cudaMemcpyAsync(flat.data(), e->flat, flat.size() * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    std::memcpy(W1, flat.data(), kTableFloats * sizeof(float));
    std::memcpy(b1, flat.data() + kTableFloats, kHidden * sizeof(float));
    std::memcpy(w2, flat.data() + kTableFloats + kHidden, kHidden * sizeof(float));
    b2[0] = flat[kTableFloats + 2 * kHidden];
    return BGX_OK;
}

// ------------------------------------------------------------------------ enumeration

static int ensure_uniq_tables(bgx_engine *e)
{
    if (e->uniq_tables) return BGX_OK;
    int per_sm = 1;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_enumerate_summary, kGameThreads, 0));
    if (per_sm < 1) per_sm = 1;
    if (per_sm > 2) per_sm = 2;
    e->uniq_grid = e->sm_count * per_sm;
    const size_t bytes = (size_t)e->uniq_grid * kGameWarps * kUniqBytesPerWarp;
    CU(cudaMalloc(&e->uniq_tables, bytes));
    CU(cudaMemsetAsync(e->uniq_tables, 0, bytes, e->stream));
    CU(cudaMalloc(&e->uniq_gens, (size_t)e->uniq_grid * kGameWarps * sizeof(uint32_t)));
    CU(cudaMemsetAsync(e->uniq_gens, 0, (size_t)e->uniq_grid * kGameWarps * sizeof(uint32_t), e->stream));
    return BGX_OK;
}

int bgx_enumerate_summary(bgx_engine *e, const int8_t *queries, int64_t n, int32_t *n_seq, int32_t *n_unique, uint64_t *digest)
{
    USE(e);
    NEED(queries && n_seq && n_unique && digest && n >= 0, "bad argument");
    int rc = ensure_uniq_tables(e);
    if (rc) return rc;
    if (n == 0) return BGX_OK;
    CU(cudaMemsetAsync(e->counter, 0, sizeof(unsigned long long), e->stream));
    tick(e);
    k_enumerate_summary<<<e->uniq_grid, kGameThreads, 0, e->stream>>>(queries, n, n_seq, n_unique,
                                                                       (unsigned long long *)digest, e->uniq_tables, e->uniq_gens, e->counter);
    tock(e);
    e->launches++;
    CU(cudaGetLastError());
    return BGX_OK;
}

int bgx_enumerate_summary_host(bgx_engine *e, const int8_t *queries, int64_t n, int32_t *n_seq, int32_t *n_unique, uint64_t *digest)
{
    USE(e);
    NEED(queries && n_seq && n_unique && digest && n >= 0, "bad argument");
    if (n == 0) return BGX_OK;
    void *dq, *dn, *du, *dd;
    int rc;
    if ((rc = scratch(e, 0, (size_t)n * 32, &dq))) return rc;
    if ((rc = scratch(e, 1, (size_t)n * 4, &dn))) return rc;
    if ((rc = scratch(e, 2, (size_t)n * 4, &du))) return rc;
    if ((rc = scratch(e, 3, (size_t)n * 8, &dd))) return rc;
    CU(cudaMemcpyAsync(dq, queries, (size_t)n * 32, cudaMemcpyHostToDevice, e->stream));
    if ((rc = bgx_enumerate_summary(e, (const int8_t *)dq, n, (int32_t *)dn, (int32_t *)du, (uint64_t *)dd))) return rc;
    CU(cudaMemcpyAsync(n_seq, dn, (size_t)n * 4, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaMemcpyAsync(n_unique, du, (size_t)n * 4, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaMemcpyAsync(digest, dd, (size_t)n * 8, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    return BGX_OK;
}

int bgx_enumerate(bgx_engine *e, const int8_t *queries, int64_t n, const int64_t *offsets,
                  int8_t *seq_moves, int8_t *seq_len, int8_t *states)
{
    USE(e);
    NEED(queries && offsets && seq_moves && seq_len && states && n >= 0, "bad argument");
    if (n == 0) return BGX_OK;
    CU(cudaMemsetAsync(e->counter, 0, sizeof(unsigned long long), e->stream));
    tick(e);
    k_enumerate_write<<<e->sm_count * 2, kGameThreads, 0, e->stream>>>(queries, n, (const long long *)offsets,
                                                                        seq_moves, seq_len, states, e->counter);
    tock(e);
    e->launches++;
    CU(cudaGetLastError());
    return BGX_OK;
}

// sizes of every query's sequence list and their exclusive prefix sum, on the device: the allocation pass of the
// materialised enumeration (a count-only walk, no dedup table, no digest) + a three-launch scan
int bgx_enumerate_count(bgx_engine *e, const int8_t *queries, int64_t n, int32_t *n_seq, int64_t *offsets)
{
    USE(e);
    NEED(queries && n_seq && offsets && n >= 0, "bad argument");
    if (n == 0) { CU(cudaMemsetAsync(offsets, 0, 8, e->stream)); return BGX_OK; }
    const int n_tiles = (int)((n + kScanTile - 1) / kScanTile);
    void *sums;
    int rc;
    if ((rc = scratch(e, 9, (size_t)(n_tiles + 1) * 8, &sums))) return rc;
    CU(cudaMemsetAsync(e->counter, 0, sizeof(unsigned long long), e->stream));
    tick(e);
    k_enumerate_count<<<e->sm_count * 2, kGameThreads, 0, e->stream>>>(queries, n, n_seq, e->counter);
    tock(e);
    k_scan_tiles<<<n_tiles, kScanThreads, 0, e->stream>>>(n_seq, n, (long long *)offsets, (long long *)sums);
    k_scan_sums<<<1, 1024, 0, e->stream>>>((long long *)sums, n_tiles);
    k_scan_add<<<(unsigned)((n + kScanThreads - 1) / kScanThreads), kScanThreads, 0, e->stream>>>((long long *)offsets, n, (const long long *)sums, n_tiles);
    e->launches += 4;
    CU(cudaGetLastError());
    return BGX_OK;
}

int bgx_enumerate_host(bgx_engine *e, const int8_t *queries, int64_t n, int64_t cap, int64_t *offsets,
                       int8_t *seq_moves, int8_t *seq_len, int8_t *states, int64_t *total)
{
    USE(e);
    NEED(queries && total && n >= 0 && cap >= 0, "bad argument");
    *total = 0;
    if (n == 0) { if (offsets) offsets[0] = 0; return BGX_OK; }
    void *dq, *dn, *doff;
    int rc;
    if ((rc = scratch(e, 0, (size_t)n * 32, &dq))) return rc;
    if ((rc = scratch(e, 1, (size_t)n * 4, &dn))) return rc;
    if ((rc = scratch(e, 4, (size_t)(n + 1) * 8, &doff))) return rc;
    CU(cudaMemcpyAsync(dq, queries, (size_t)n * 32, cudaMemcpyHostToDevice, e->stream));
    if ((rc = bgx_enumerate_count(e, (const int8_t *)dq, n, (int32_t *)dn, (int64_t *)doff))) return rc;
    // the one number the host needs before it can size anything: 8 bytes
    int64_t rows_needed = 0;
    CU(cudaMemcpyAsync(&rows_needed, (const int64_t *)doff + n, 8, cudaMemcpyDeviceToHost, e->stream));
    if (offsets) CU(cudaMemcpyAsync(offsets, doff, (size_t)(n + 1) * 8, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    *total = rows_needed;
    if (rows_needed > cap) { set_error("bgx_enumerate_host: %lld rows needed, cap %lld", (long long)rows_needed, (long long)cap); return BGX_E_CAPACITY; }
    NEED(seq_moves && seq_len && states, "null output buffer");
    const size_t rows = (size_t)rows_needed;
    if (rows == 0) return BGX_OK;
    void *dm, *dl, *ds;
    if ((rc = scratch(e, 5, rows * 8, &dm))) return rc;
    if ((rc = scratch(e, 6, rows, &dl))) return rc;
    if ((rc = scratch(e, 7, rows * 32, &ds))) return rc;
    if ((rc = bgx_enumerate(e, (const int8_t *)dq, n, (const int64_t *)doff, (int8_t *)dm, (int8_t *)dl, (int8_t *)ds))) return rc;
    CU(cudaMemcpyAsync(seq_moves, dm, rows * 8, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaMemcpyAsync(seq_len, dl, rows, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaMemcpyAsync(states, ds, rows * 32, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    return BGX_OK;
}

// ------------------------------------------------------------------------ encode / evaluate

int bgx_encode(bgx_engine *e, const int8_t *records, int64_t n, float *X)
{
    USE(e);
    NEED(records && X && n >= 0, "bad argument");
    NEED(((uintptr_t)X & 15) == 0 && ((uintptr_t)records & 3) == 0, "X must be 16-byte aligned, records 4-byte aligned");
    if (n == 0) return BGX_OK;
    const long long tiles = (n + kEncRows - 1) / kEncRows;
    long long grid = (long long)e->sm_count * 4;     // 4 CTAs of 2 x 25 KB tiles are resident per SM
    if (grid > tiles) grid = tiles;
    tick(e);
    k_encode<<<(int)grid, kEncWarps * 32, kEncSmem, e->stream>>>(records, n, X);
    tock(e);
    e->launches++;
    CU(cudaGetLastError());
    return BGX_OK;
}

int bgx_encode_host(bgx_engine *e, const int8_t *records, int64_t n, float *X)
{
    USE(e);
    NEED(records && X && n >= 0, "bad argument");
    if (n == 0) return BGX_OK;
    void *dq, *dx;
    int rc;
    if ((rc = scratch(e, 0, (size_t)n * 32, &dq))) return rc;
    if ((rc = scratch(e, 8, (size_t)n * kFeatures * 4, &dx))) return rc;
    CU(cudaMemcpyAsync(dq, records, (size_t)n * 32, cudaMemcpyHostToDevice, e->stream));
    if ((rc = bgx_encode(e, (const int8_t *)dq, n, (float *)dx))) return rc;
    CU(cudaMemcpyAsync(X, dx, (size_t)n * kFeatures * 4, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    return BGX_OK;
}

int bgx_evaluate(bgx_engine *e, const int8_t *records, int64_t n, float *V)
{
    USE(e);
    NEED(records && V && n >= 0, "bad argument");
    if (!e->have_weights) { set_error("bgx_evaluate: weights not set"); return BGX_E_STATE; }
    if (n == 0) return BGX_OK;
    tick(e);
    k_evaluate<<<game_grid(e), kGameThreads, kEvalSmem, e->stream>>>(records, n, V, e->fixed, e->flat);
    tock(e);
    e->launches++;
    CU(cudaGetLastError());
    return BGX_OK;
}

int bgx_evaluate_host(bgx_engine *e, const int8_t *records, int64_t n, float *V)
{
    USE(e);
    NEED(records && V && n >= 0, "bad argument");
    if (n == 0) return BGX_OK;
    void *dq, *dv;
    int rc;
    if ((rc = scratch(e, 0, (size_t)n * 32, &dq))) return rc;
    if ((rc = scratch(e, 1, (size_t)n * 4, &dv))) return rc;
    CU(cudaMemcpyAsync(dq, records, (size_t)n * 32, cudaMemcpyHostToDevice, e->stream));
    if ((rc = bgx_evaluate(e, (const int8_t *)dq, n, (float *)dv))) return rc;
    CU(cudaMemcpyAsync(V, dv, (size_t)n * 4, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    return BGX_OK;
}

// ------------------------------------------------------------------------ batched make_move

// the sorted queue of one launch: read from `slot` (computed here by k_select_order unless the previous launch of the lane left
// it there), and - in the fused play-ply form - the next launch's queue written to the other slot
struct OrderPlan {
    int32_t *region[2] = {nullptr, nullptr};
    int slot = 0;
    bool ready = false;          // region[slot] / totals[slot] were produced by the previous launch
    bool produce = false;        // fill region[1 - slot] for the next launch (adv.next must be set)
};

static int launch_select(bgx_engine *e, cudaStream_t stream, unsigned long long *counter, StealResult *steal,
                         const int8_t *queries, int64_t n, float epsilon, uint64_t seed, const SelectOut &out, const OrderPlan &plan,
                         int grid = 0, AdvanceOut adv = AdvanceOut{})
{
    if (grid <= 0 || grid > e->sm_count) grid = game_grid(e);
    uint32_t *totals_of[2] = {reinterpret_cast<uint32_t *>(counter) + 16, reinterpret_cast<uint32_t *>(counter) + 32};
    int32_t *region = plan.region[plan.slot];
    uint32_t *totals = totals_of[plan.slot];
    CU(cudaMemsetAsync(counter, 0, sizeof(unsigned long long), stream));
    if (region && !plan.ready) {
        CU(cudaMemsetAsync(totals, 0, kOrderBuckets * sizeof(uint32_t), stream));
        k_select_order<<<(unsigned)((n + kOrderCtaQueries - 1) / kOrderCtaQueries), 256, 0, stream>>>(queries, n, region, totals);
        e->launches++;
    }
    adv.next_region = nullptr;
    adv.next_totals = nullptr;
    if (plan.produce && adv.next && plan.region[1 - plan.slot]) {
        adv.next_region = plan.region[1 - plan.slot];
        adv.next_totals = totals_of[1 - plan.slot];
        CU(cudaMemsetAsync(adv.next_totals, 0, kOrderBuckets * sizeof(uint32_t), stream));
    }
    const SelectTune tune = {(unsigned long long)(n * (int64_t)e->select_urgent_from_pct / 100), e->select_urgent_min, e->select_giant_min};
#define BGX_LAUNCH_SELECT(W, S, X)                                                                          \
    k_select<W, S, X><<<grid, W * 32, ply_smem<W, S>(), stream>>>(queries, n, epsilon, (uint32_t)seed, \
                                                                          (uint32_t)(seed >> 32), out, e->fixed, e->flat, counter, steal, tune, region, totals, adv)
    const bool ex = epsilon > 0.f;
    if (e->select_warps == 16) { if (ex) BGX_LAUNCH_SELECT(16, 109, true); else BGX_LAUNCH_SELECT(16, 109, false); }
    else if (e->select_warps == 20) { if (ex) BGX_LAUNCH_SELECT(20, 86, true); else BGX_LAUNCH_SELECT(20, 86, false); }
    else if (e->select_warps == 24) { if (ex) BGX_LAUNCH_SELECT(24, 72, true); else BGX_LAUNCH_SELECT(24, 72, false); }
    else { if (ex) BGX_LAUNCH_SELECT(32, 53, true); else BGX_LAUNCH_SELECT(32, 53, false); }
#undef BGX_LAUNCH_SELECT
    e->launches++;
    CU(cudaGetLastError());
    return BGX_OK;
}

int bgx_select_moves(bgx_engine *e, const int8_t *queries, int64_t n, float epsilon, uint64_t seed,
                     int8_t *chosen, int8_t *moves, int8_t *moves_len, float *value, int32_t *n_seq, int32_t *n_scored)
{
    USE(e);
    NEED(queries && n >= 0, "bad argument");
    if (!e->have_weights) { set_error("bgx_select_moves: weights not set"); return BGX_E_STATE; }
    if (n == 0) return BGX_OK;
    const SelectOut out = {chosen, moves, moves_len, value, n_seq, n_scored};
    void *region = nullptr;
    if (n <= e->select_order_max) {
        const int rs = scratch(e, 11, (size_t)n * kOrderBuckets * 4, &region);
        if (rs) return rs;
    }
    OrderPlan plan;
    plan.region[0] = (int32_t *)region;
    tick(e);
    const int rc = launch_select(e, e->stream, e->counter, e->steal, queries, n, epsilon, seed, out, plan);
    tock(e);
    return rc;
}

int bgx_select_moves_host(bgx_engine *e, const int8_t *queries, int64_t n, float epsilon, uint64_t seed,
                          int8_t *chosen, int8_t *moves, int8_t *moves_len, float *value, int32_t *n_seq, int32_t *n_scored)
{
    USE(e);
    NEED(queries && n >= 0, "bad argument");
    if (n == 0) return BGX_OK;
    void *dq, *dc, *dm, *dl, *dv, *dn, *ds;
    int rc;
    if ((rc = scratch(e, 0, (size_t)n * 32, &dq))) return rc;
    if ((rc = scratch(e, 1, (size_t)n * 32, &dc))) return rc;
    if ((rc = scratch(e, 2, (size_t)n * 8, &dm))) return rc;
    if ((rc = scratch(e, 3, (size_t)n, &dl))) return rc;
    if ((rc = scratch(e, 4, (size_t)n * 4, &dv))) return rc;
    if ((rc = scratch(e, 5, (size_t)n * 4, &dn))) return rc;
    if ((rc = scratch(e, 6, (size_t)n * 4, &ds))) return rc;
    CU(cudaMemcpyAsync(dq, queries, (size_t)n * 32, cudaMemcpyHostToDevice, e->stream));
    rc = bgx_select_moves(e, (const int8_t *)dq, n, epsilon, seed, chosen ? (int8_t *)dc : nullptr, moves ? (int8_t *)dm : nullptr,
                          moves_len ? (int8_t *)dl : nullptr, value ? (float *)dv : nullptr,
                          n_seq ? (int32_t *)dn : nullptr, n_scored ? (int32_t *)ds : nullptr);
    if (rc) return rc;
    if (chosen) CU(cudaMemcpyAsync(chosen, dc, (size_t)n * 32, cudaMemcpyDeviceToHost, e->stream));
    if (moves) CU(cudaMemcpyAsync(moves, dm, (size_t)n * 8, cudaMemcpyDeviceToHost, e->stream));
    if (moves_len) CU(cudaMemcpyAsync(moves_len, dl, (size_t)n, cudaMemcpyDeviceToHost, e->stream));
    if (value) CU(cudaMemcpyAsync(value, dv, (size_t)n * 4, cudaMemcpyDeviceToHost, e->stream));
    if (n_seq) CU(cudaMemcpyAsync(n_seq, dn, (size_t)n * 4, cudaMemcpyDeviceToHost, e->stream));
    if (n_scored) CU(cudaMemcpyAsync(n_scored, ds, (size_t)n * 4, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    return BGX_OK;
}

// ------------------------------------------------------------------------ two-ply move selection (DESIGN 7c)

constexpr long long kTwoplyChunk = 1ll << 21;   // replies per k_select launch: the sorted-queue limit (select_order_max default)

// with "twoply_timing": the time since the previous mark goes to stage k (0 candidates, 1 expand, 2 replies, 3 reduce)
static int twoply_mark(bgx_engine *e, int k)
{
    if (!e->twoply_timing) return BGX_OK;
    CU(cudaEventRecord(e->tp1, e->stream));
    CU(cudaEventSynchronize(e->tp1));
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, e->tp0, e->tp1));
    e->twoply_ms[k] += ms;
    CU(cudaEventRecord(e->tp0, e->stream));
    return BGX_OK;
}
#define TWOPLY_MARK(e, k) do { const int rc__ = twoply_mark(e, k); if (rc__ != BGX_OK) return rc__; } while (0)

// exclusive prefix sum of cnt[n] into offsets[n + 1] (the k_scan_* launches of bgx_enumerate_count)
static int scan_counts(bgx_engine *e, const int32_t *cnt, int64_t n, long long *offsets, long long *sums)
{
    const int n_tiles = (int)((n + kScanTile - 1) / kScanTile);
    k_scan_tiles<<<n_tiles, kScanThreads, 0, e->stream>>>(cnt, n, offsets, sums);
    k_scan_sums<<<1, 1024, 0, e->stream>>>(sums, n_tiles);
    k_scan_add<<<(unsigned)((n + kScanThreads - 1) / kScanThreads), kScanThreads, 0, e->stream>>>(offsets, n, sums, n_tiles);
    e->launches += 3;
    CU(cudaGetLastError());
    return BGX_OK;
}

int bgx_select_moves_2ply(bgx_engine *e, const int8_t *queries, int64_t n, int32_t max_candidates,
                          int8_t *chosen, int8_t *moves, int8_t *moves_len, float *value, int32_t *n_candidates, int32_t *n_expanded)
{
    USE(e);
    NEED(queries && n >= 0 && max_candidates >= 0, "bad argument");
    if (!e->have_weights) { set_error("bgx_select_moves_2ply: weights not set"); return BGX_E_STATE; }
    if (n == 0) return BGX_OK;
    int rc = ensure_uniq_tables(e);
    if (rc) return rc;
    if (e->twoply_timing) {
        if (!e->tp0) { CU(cudaEventCreate(&e->tp0)); CU(cudaEventCreate(&e->tp1)); }
        CU(cudaEventRecord(e->tp0, e->stream));
    }
    const int n_tiles = (int)((n + kScanTile - 1) / kScanTile);
    void *d_nseq, *d_u, *d_dig, *d_cnt, *d_off, *d_sums, *d_flags, *d_nexp, *d_eoff;
    if ((rc = scratch(e, 12, (size_t)n * 4, &d_nseq))) return rc;
    if ((rc = scratch(e, 13, (size_t)n * 4, &d_u))) return rc;
    if ((rc = scratch(e, 14, (size_t)n * 8, &d_dig))) return rc;
    if ((rc = scratch(e, 15, (size_t)n * 4, &d_cnt))) return rc;
    if ((rc = scratch(e, 16, (size_t)(n + 1) * 8, &d_off))) return rc;
    if ((rc = scratch(e, 17, (size_t)(n_tiles + 1) * 8, &d_sums))) return rc;
    if ((rc = scratch(e, 18, 16, &d_flags))) return rc;
    if ((rc = scratch(e, 19, (size_t)n * 4, &d_nexp))) return rc;
    if ((rc = scratch(e, 20, (size_t)(n + 1) * 8, &d_eoff))) return rc;
    int32_t *cnt = (int32_t *)d_cnt, *nexp = (int32_t *)d_nexp;
    long long *off = (long long *)d_off, *eoff = (long long *)d_eoff, *sums = (long long *)d_sums;
    int *flags = (int *)d_flags;

    // 1. candidates: U per query (the summary walk), their offsets, then every distinct afterstate with its first sequence and V
    CU(cudaMemsetAsync(flags, 0, 16, e->stream));
    CU(cudaMemsetAsync(e->counter, 0, sizeof(unsigned long long), e->stream));
    k_enumerate_summary<<<e->uniq_grid, kGameThreads, 0, e->stream>>>(queries, n, (int32_t *)d_nseq, (int32_t *)d_u,
                                                                       (unsigned long long *)d_dig, e->uniq_tables, e->uniq_gens, e->counter);
    k_twoply_count<<<(unsigned)((n + 255) / 256), 256, 0, e->stream>>>((const int32_t *)d_u, n, cnt, flags);
    e->launches += 2;
    if ((rc = scan_counts(e, cnt, n, off, sums))) return rc;
    long long n_cand = 0;
    int hflags[4] = {};
    CU(cudaMemcpyAsync(&n_cand, off + n, 8, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaMemcpyAsync(hflags, flags, 16, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    if (hflags[0]) {
        set_error("bgx_select_moves_2ply: a query has more distinct afterstates than the exact-dedup table holds (%d)", kUniqSlots);
        return BGX_E_CAPACITY;
    }
    void *d_rec = nullptr, *d_mv = nullptr, *d_len = nullptr, *d_val = nullptr, *d_exp = nullptr, *d_e2 = nullptr;
    const size_t C = (size_t)(n_cand > 0 ? n_cand : 1);
    if ((rc = scratch(e, 21, C * 32, &d_rec))) return rc;
    if ((rc = scratch(e, 22, C * 8, &d_mv))) return rc;
    if ((rc = scratch(e, 23, C, &d_len))) return rc;
    if ((rc = scratch(e, 24, C * 4, &d_val))) return rc;
    if ((rc = scratch(e, 25, C, &d_exp))) return rc;
    if ((rc = scratch(e, 26, C * 4, &d_e2))) return rc;
    int8_t *rec = (int8_t *)d_rec, *cmv = (int8_t *)d_mv, *clen = (int8_t *)d_len, *expand = (int8_t *)d_exp;
    float *val = (float *)d_val, *e2 = (float *)d_e2;
    if (n_cand > 0) {
        CU(cudaMemsetAsync(e->counter, 0, sizeof(unsigned long long), e->stream));
        k_candidates<<<game_grid(e), kGameThreads, kEvalSmem, e->stream>>>(queries, n, cnt, off, rec, cmv, clen, val, e->uniq_tables,
                                                                           e->uniq_gens, e->counter, flags, e->fixed);
        e->launches++;
        CU(cudaGetLastError());
    }
    TWOPLY_MARK(e, 0);

    // 2. which candidates are expanded, and the list of them
    const unsigned small_grid = (unsigned)std::min<long long>((n + 7) / 8, (long long)e->sm_count * 8);
    k_twoply_expand<<<small_grid, 256, 0, e->stream>>>(queries, n, cnt, off, rec, val, max_candidates, expand, nexp);
    e->launches++;
    if ((rc = scan_counts(e, nexp, n, eoff, sums))) return rc;
    long long n_exp = 0;
    CU(cudaMemcpyAsync(&n_exp, eoff + n, 8, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaMemcpyAsync(hflags, flags, 16, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    if (hflags[0] & 2) {
        set_error("bgx_select_moves_2ply: the candidate walk disagreed with the summary walk");
        return BGX_E_CUDA;
    }
    void *d_list = nullptr;
    if ((rc = scratch(e, 27, (size_t)(n_exp > 0 ? n_exp : 1) * 8, &d_list))) return rc;
    long long *list = (long long *)d_list;
    if (n_exp > 0) {
        k_twoply_list<<<small_grid, 256, 0, e->stream>>>(n, cnt, off, expand, eoff, list);
        e->launches++;
    }
    TWOPLY_MARK(e, 1);

    // 3. replies in chunks: 21 records per expanded candidate, k_select (values only), the expectation
    const long long chunk_replies = std::max<long long>(e->twoply_chunk > 0 ? e->twoply_chunk : kTwoplyChunk, kRolls);
    const long long per_chunk = chunk_replies / kRolls;
    const long long cap_replies = std::min<long long>(n_exp, per_chunk) * kRolls;
    void *d_rep = nullptr, *d_rval = nullptr, *region = nullptr;
    if (n_exp > 0) {
        if ((rc = scratch(e, 28, (size_t)cap_replies * 32, &d_rep))) return rc;
        if ((rc = scratch(e, 29, (size_t)cap_replies * 4, &d_rval))) return rc;
        if (cap_replies <= e->select_order_max && (rc = scratch(e, 30, (size_t)cap_replies * kOrderBuckets * 4, &region))) return rc;
    }
    for (long long e0 = 0; e0 < n_exp; e0 += per_chunk) {
        const long long e1 = std::min(n_exp, e0 + per_chunk);
        const long long nr = (e1 - e0) * kRolls;
        k_twoply_replies<<<(unsigned)std::min<long long>((nr + 7) / 8, (long long)e->sm_count * 16), 256, 0, e->stream>>>(list, e0, nr, rec,
                                                                                                                        (int8_t *)d_rep);
        e->launches++;
        const SelectOut out = {nullptr, nullptr, nullptr, (float *)d_rval, nullptr, nullptr};
        OrderPlan plan;
        plan.region[0] = nr <= e->select_order_max ? (int32_t *)region : nullptr;
        if ((rc = launch_select(e, e->stream, e->counter, e->steal, (const int8_t *)d_rep, nr, 0.f, 0, out, plan))) return rc;
        TWOPLY_MARK(e, 2);
        k_twoply_reduce<<<game_grid(e), kGameThreads, kEvalSmem, e->stream>>>(list, e0, e1, rec, (const float *)d_rval, e2, e->fixed);
        e->launches++;
        CU(cudaGetLastError());
        TWOPLY_MARK(e, 3);
    }

    // 4. the pick
    k_twoply_pick<<<small_grid, 256, 0, e->stream>>>(queries, n, cnt, off, rec, cmv, clen, expand, e2, nexp, chosen, moves, moves_len, value,
                                                     n_candidates, n_expanded);
    e->launches++;
    CU(cudaGetLastError());
    TWOPLY_MARK(e, 3);
    return BGX_OK;
}

int bgx_select_moves_2ply_host(bgx_engine *e, const int8_t *queries, int64_t n, int32_t max_candidates,
                               int8_t *chosen, int8_t *moves, int8_t *moves_len, float *value, int32_t *n_candidates, int32_t *n_expanded)
{
    USE(e);
    NEED(queries && n >= 0 && max_candidates >= 0, "bad argument");
    if (!e->have_weights) { set_error("bgx_select_moves_2ply_host: weights not set"); return BGX_E_STATE; }
    if (n == 0) return BGX_OK;
    void *dq, *dc, *dm, *dl, *dv, *dn, *dx;
    int rc;
    if ((rc = scratch(e, 0, (size_t)n * 32, &dq))) return rc;
    if ((rc = scratch(e, 1, (size_t)n * 32, &dc))) return rc;
    if ((rc = scratch(e, 2, (size_t)n * 8, &dm))) return rc;
    if ((rc = scratch(e, 3, (size_t)n, &dl))) return rc;
    if ((rc = scratch(e, 4, (size_t)n * 4, &dv))) return rc;
    if ((rc = scratch(e, 5, (size_t)n * 4, &dn))) return rc;
    if ((rc = scratch(e, 6, (size_t)n * 4, &dx))) return rc;
    CU(cudaMemcpyAsync(dq, queries, (size_t)n * 32, cudaMemcpyHostToDevice, e->stream));
    rc = bgx_select_moves_2ply(e, (const int8_t *)dq, n, max_candidates, chosen ? (int8_t *)dc : nullptr, moves ? (int8_t *)dm : nullptr,
                               moves_len ? (int8_t *)dl : nullptr, value ? (float *)dv : nullptr,
                               n_candidates ? (int32_t *)dn : nullptr, n_expanded ? (int32_t *)dx : nullptr);
    if (rc) return rc;
    if (chosen) CU(cudaMemcpyAsync(chosen, dc, (size_t)n * 32, cudaMemcpyDeviceToHost, e->stream));
    if (moves) CU(cudaMemcpyAsync(moves, dm, (size_t)n * 8, cudaMemcpyDeviceToHost, e->stream));
    if (moves_len) CU(cudaMemcpyAsync(moves_len, dl, (size_t)n, cudaMemcpyDeviceToHost, e->stream));
    if (value) CU(cudaMemcpyAsync(value, dv, (size_t)n * 4, cudaMemcpyDeviceToHost, e->stream));
    if (n_candidates) CU(cudaMemcpyAsync(n_candidates, dn, (size_t)n * 4, cudaMemcpyDeviceToHost, e->stream));
    if (n_expanded) CU(cudaMemcpyAsync(n_expanded, dx, (size_t)n * 4, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    return BGX_OK;
}

int bgx_twoply_stage_ms(bgx_engine *e, double *ms)
{
    if (!e || !ms) { set_error("bgx_twoply_stage_ms: null"); return BGX_E_INVALID; }
    for (int k = 0; k < 4; k++) { ms[k] = e->twoply_ms[k]; e->twoply_ms[k] = 0.0; }
    return BGX_OK;
}

// ------------------------------------------------------------------------ rollouts (DESIGN 7d)

constexpr long long kRolloutChunk = 1ll << 24;  // trials per k_rollout launch: 36 MB of per-trial scratch

static int rollout_args(int64_t n, int32_t trials, int32_t max_plies, int flags, const char *who)
{
    if (n < 0 || trials < 1) { set_error("%s: n must be >= 0 and trials >= 1", who); return BGX_E_INVALID; }
    if (max_plies < 0 || max_plies > BGX_ROLLOUT_MAX_PLIES) { set_error("%s: max_plies must be 0 .. %d", who, BGX_ROLLOUT_MAX_PLIES); return BGX_E_INVALID; }
    if (flags & ~BGX_ROLLOUT_STRATIFY) { set_error("%s: unknown flags 0x%x", who, flags); return BGX_E_INVALID; }
    if ((flags & BGX_ROLLOUT_STRATIFY) && trials % 36 != 0) { set_error("%s: a stratified rollout needs a multiple of 36 trials", who); return BGX_E_INVALID; }
    return BGX_OK;
}

int bgx_rollout(bgx_engine *e, const int8_t *positions, int64_t n, int32_t trials, int32_t max_plies, uint64_t seed, int flags,
                double *mean, double *std_err, int64_t *counts, float *trial_value, int8_t *trial_outcome, int32_t *trial_plies)
{
    USE(e);
    if (int rc = rollout_args(n, trials, max_plies, flags, "bgx_rollout")) return rc;
    NEED(positions || n == 0, "null positions");
    if (!e->have_weights) { set_error("bgx_rollout: weights not set"); return BGX_E_STATE; }
    if (n == 0) return BGX_OK;
    // chunks of whole positions; the per-trial results of a chunk go to the caller's arrays or to engine scratch
    const long long chunk = e->rollout_chunk > 0 ? e->rollout_chunk : kRolloutChunk;
    const long long per_launch = std::max<long long>(1, chunk / trials);
    const long long items_cap = std::min<long long>(n, per_launch) * trials;
    void *sv = nullptr, *so = nullptr, *sp = nullptr;
    int rc;
    if (!trial_value && (rc = scratch(e, 32, (size_t)items_cap * 4, &sv))) return rc;
    if (!trial_outcome && (rc = scratch(e, 33, (size_t)items_cap, &so))) return rc;
    if (!trial_plies && (rc = scratch(e, 34, (size_t)items_cap * 4, &sp))) return rc;
    RolloutParams p;
    p.trials = trials;
    p.cap = max_plies > 0 ? max_plies : BGX_ROLLOUT_MAX_PLIES;
    p.stratify = (flags & BGX_ROLLOUT_STRATIFY) ? 1 : 0;
    p.seed_lo = (uint32_t)seed; p.seed_hi = (uint32_t)(seed >> 32);
    p.counter = e->counter; p.zstash = e->zstash;
    tick(e);
    for (long long q0 = 0; q0 < n; q0 += per_launch) {
        const long long np = std::min<long long>(n - q0, per_launch);
        const size_t at = (size_t)q0 * trials;
        p.positions = positions + q0 * 32;
        p.n_items = np * trials;
        p.value = trial_value ? trial_value + at : (float *)sv;
        p.outcome = trial_outcome ? trial_outcome + at : (int8_t *)so;
        p.plies = trial_plies ? trial_plies + at : (int32_t *)sp;
        CU(cudaMemsetAsync(e->counter, 0, sizeof(unsigned long long), e->stream));
#define BGX_LAUNCH_ROLLOUT(W, S) k_rollout<W, S><<<game_grid(e), W * 32, ply_smem<W, S>(), e->stream>>>(p, e->fixed, e->steal)
        if (e->rollout_warps == 16) BGX_LAUNCH_ROLLOUT(16, 109);
        else if (e->rollout_warps == 20) BGX_LAUNCH_ROLLOUT(20, 86);
        else if (e->rollout_warps == 24) BGX_LAUNCH_ROLLOUT(24, 72);
        else BGX_LAUNCH_ROLLOUT(32, 53);
#undef BGX_LAUNCH_ROLLOUT
        if (mean || std_err || counts)
            k_rollout_reduce<<<(unsigned)((np + 127) / 128), 128, 0, e->stream>>>(p.value, p.outcome, p.plies, np, trials, mean ? mean + q0 : nullptr,
                                                                              std_err ? std_err + q0 : nullptr,
                                                                              counts ? (long long *)counts + q0 * 8 : nullptr);
        e->launches += 2;
        CU(cudaGetLastError());
    }
    tock(e);
    return BGX_OK;
}

int bgx_rollout_host(bgx_engine *e, const int8_t *positions, int64_t n, int32_t trials, int32_t max_plies, uint64_t seed, int flags,
                     double *mean, double *std_err, int64_t *counts, float *trial_value, int8_t *trial_outcome, int32_t *trial_plies)
{
    USE(e);
    if (int rc = rollout_args(n, trials, max_plies, flags, "bgx_rollout_host")) return rc;
    NEED(positions || n == 0, "null positions");
    if (!e->have_weights) { set_error("bgx_rollout_host: weights not set"); return BGX_E_STATE; }
    if (n == 0) return BGX_OK;
    const size_t items = (size_t)n * trials;
    void *dq, *dm = nullptr, *ds = nullptr, *dc = nullptr, *dv = nullptr, *dout = nullptr, *dp = nullptr;
    int rc;
    if ((rc = scratch(e, 35, (size_t)n * 32, &dq))) return rc;
    if (mean && (rc = scratch(e, 36, (size_t)n * 8, &dm))) return rc;
    if (std_err && (rc = scratch(e, 37, (size_t)n * 8, &ds))) return rc;
    if (counts && (rc = scratch(e, 38, (size_t)n * 64, &dc))) return rc;
    if (trial_value && (rc = scratch(e, 39, items * 4, &dv))) return rc;
    if (trial_outcome && (rc = scratch(e, 0, items, &dout))) return rc;
    if (trial_plies && (rc = scratch(e, 1, items * 4, &dp))) return rc;
    CU(cudaMemcpyAsync(dq, positions, (size_t)n * 32, cudaMemcpyHostToDevice, e->stream));
    if ((rc = bgx_rollout(e, (const int8_t *)dq, n, trials, max_plies, seed, flags, (double *)dm, (double *)ds, (int64_t *)dc,
                          (float *)dv, (int8_t *)dout, (int32_t *)dp))) return rc;
    if (mean) CU(cudaMemcpyAsync(mean, dm, (size_t)n * 8, cudaMemcpyDeviceToHost, e->stream));
    if (std_err) CU(cudaMemcpyAsync(std_err, ds, (size_t)n * 8, cudaMemcpyDeviceToHost, e->stream));
    if (counts) CU(cudaMemcpyAsync(counts, dc, (size_t)n * 64, cudaMemcpyDeviceToHost, e->stream));
    if (trial_value) CU(cudaMemcpyAsync(trial_value, dv, items * 4, cudaMemcpyDeviceToHost, e->stream));
    if (trial_outcome) CU(cudaMemcpyAsync(trial_outcome, dout, items, cudaMemcpyDeviceToHost, e->stream));
    if (trial_plies) CU(cudaMemcpyAsync(trial_plies, dp, items * 4, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    return BGX_OK;
}

// Asynchronous form of bgx_select_moves_host: the copies and the kernel are queued on lane `lane`'s own
// stream and the call returns; bgx_lane_wait blocks until that lane's results are in the host buffers.
// A few lanes in flight let the host advance one part of a population while the GPU plays the others.
static int lane_scratch(bgx_lane &l, int i, size_t bytes, void **out)
{
    if (l.cap[i] < bytes) {
        if (l.buf[i]) CU(cudaFree(l.buf[i]));
        l.buf[i] = nullptr;
        l.cap[i] = 0;
        const size_t want = bytes + bytes / 4 + 256;
        CU(cudaMalloc(&l.buf[i], want));
        l.cap[i] = want;
    }
    *out = l.buf[i];
    return BGX_OK;
}

int bgx_select_moves_host_async(bgx_engine *e, int lane, const int8_t *queries, int64_t n, float epsilon, uint64_t seed,
                                int8_t *chosen, int8_t *moves, int8_t *moves_len, float *value, int32_t *n_seq, int32_t *n_scored)
{
    USE(e);
    NEED(lane >= 0 && lane < kLanes, "lane out of range");
    NEED(queries && n >= 0, "bad argument");
    if (!e->have_weights) { set_error("bgx_select_moves_host_async: weights not set"); return BGX_E_STATE; }
    bgx_lane &l = e->lanes[lane];
    if (l.busy) { set_error("bgx_select_moves_host_async: lane %d has a batch in flight (bgx_lane_wait first)", lane); return BGX_E_STATE; }
    if (!l.stream) {
        CU(cudaStreamCreateWithFlags(&l.stream, cudaStreamNonBlocking));
        CU(cudaEventCreateWithFlags(&l.done, cudaEventDisableTiming));
        CU(cudaMalloc(&l.counter, kCounterBytes));
        CU(cudaMalloc(&l.steal, (size_t)e->sm_count * 32 * kStealMaxResults * sizeof(StealResult)));
    }
    if (n == 0) return BGX_OK;
    void *dq, *dc, *dm, *dl, *dv, *dn, *ds;
    int rc;
    if ((rc = lane_scratch(l, 0, (size_t)n * 32, &dq))) return rc;
    if ((rc = lane_scratch(l, 1, (size_t)n * 32, &dc))) return rc;
    if ((rc = lane_scratch(l, 2, (size_t)n * 8, &dm))) return rc;
    if ((rc = lane_scratch(l, 3, (size_t)n, &dl))) return rc;
    if ((rc = lane_scratch(l, 4, (size_t)n * 4, &dv))) return rc;
    if ((rc = lane_scratch(l, 5, (size_t)n * 4, &dn))) return rc;
    if ((rc = lane_scratch(l, 6, (size_t)n * 4, &ds))) return rc;
    // weights set on the engine's stream before this call are visible to the lane
    CU(cudaEventRecord(e->ev_sync, e->stream));
    CU(cudaStreamWaitEvent(l.stream, e->ev_sync, 0));
    CU(cudaMemcpyAsync(dq, queries, (size_t)n * 32, cudaMemcpyHostToDevice, l.stream));
    const SelectOut out = {chosen ? (int8_t *)dc : nullptr, moves ? (int8_t *)dm : nullptr, moves_len ? (int8_t *)dl : nullptr,
                           value ? (float *)dv : nullptr, n_seq ? (int32_t *)dn : nullptr, n_scored ? (int32_t *)ds : nullptr};
    void *region = nullptr;
    if (n <= e->select_order_max && (rc = lane_scratch(l, 7, (size_t)n * kOrderBuckets * 4, &region))) return rc;
    OrderPlan plan;
    plan.region[0] = (int32_t *)region;
    l.order_n = -1;
    if ((rc = launch_select(e, l.stream, l.counter, l.steal, (const int8_t *)dq, n, epsilon, seed, out, plan, e->lane_grid))) return rc;
    if (chosen) CU(cudaMemcpyAsync(chosen, dc, (size_t)n * 32, cudaMemcpyDeviceToHost, l.stream));
    if (moves) CU(cudaMemcpyAsync(moves, dm, (size_t)n * 8, cudaMemcpyDeviceToHost, l.stream));
    if (moves_len) CU(cudaMemcpyAsync(moves_len, dl, (size_t)n, cudaMemcpyDeviceToHost, l.stream));
    if (value) CU(cudaMemcpyAsync(value, dv, (size_t)n * 4, cudaMemcpyDeviceToHost, l.stream));
    if (n_seq) CU(cudaMemcpyAsync(n_seq, dn, (size_t)n * 4, cudaMemcpyDeviceToHost, l.stream));
    if (n_scored) CU(cudaMemcpyAsync(n_scored, ds, (size_t)n * 4, cudaMemcpyDeviceToHost, l.stream));
    CU(cudaEventRecord(l.done, l.stream));
    l.busy = true;
    return BGX_OK;
}

static int play_ply(bgx_engine *e, int lane, const int8_t *records, int32_t *ply, int64_t *game_id, int64_t id_stride, int first_mover,
                    int64_t n, float epsilon, uint64_t explore_seed, uint64_t dice_seed,
                    int8_t *next_records, int8_t *winner, float *value, int32_t *n_seq, const char *who)
{
    NEED(lane >= 0 && lane < kLanes, "lane out of range");
    NEED(records && next_records && n >= 0, "bad argument");
    if (!e->have_weights) { set_error("%s: weights not set", who); return BGX_E_STATE; }
    bgx_lane &l = e->lanes[lane];
    if (l.busy) { set_error("%s: lane %d has a batch in flight (bgx_lane_wait first)", who, lane); return BGX_E_STATE; }
    if (!l.stream) {
        CU(cudaStreamCreateWithFlags(&l.stream, cudaStreamNonBlocking));
        CU(cudaEventCreateWithFlags(&l.done, cudaEventDisableTiming));
        CU(cudaMalloc(&l.counter, kCounterBytes));
        CU(cudaMalloc(&l.steal, (size_t)e->sm_count * 32 * kStealMaxResults * sizeof(StealResult)));
    }
    if (n == 0) return BGX_OK;
    void *dq, *dc, *dw, *dv, *dn, *dp = nullptr, *dg = nullptr, *r0 = nullptr, *r1 = nullptr;
    int rc;
    if ((rc = lane_scratch(l, 0, (size_t)n * 32, &dq))) return rc;
    if ((rc = lane_scratch(l, 1, (size_t)n * 32, &dc))) return rc;
    if ((rc = lane_scratch(l, 3, (size_t)n, &dw))) return rc;
    if ((rc = lane_scratch(l, 4, (size_t)n * 4, &dv))) return rc;
    if ((rc = lane_scratch(l, 5, (size_t)n * 4, &dn))) return rc;
    if (ply && (rc = lane_scratch(l, 8, (size_t)n * 4, &dp))) return rc;
    if (game_id && (rc = lane_scratch(l, 9, (size_t)n * 8, &dg))) return rc;
    OrderPlan plan;
    if (n <= e->select_order_max) {
        const void *before[2] = {l.buf[7], l.buf[10]};
        if ((rc = lane_scratch(l, 7, (size_t)n * kOrderBuckets * 4, &r0))) return rc;
        if ((rc = lane_scratch(l, 10, (size_t)n * kOrderBuckets * 4, &r1))) return rc;
        if (before[0] != l.buf[7] || before[1] != l.buf[10]) l.order_n = -1;      // reallocated: the stored queue is gone
        plan.region[0] = (int32_t *)r0;
        plan.region[1] = (int32_t *)r1;
        plan.slot = l.order_slot;
        plan.ready = l.order_n == n;           // the previous call on this lane sorted ITS outputs for us: if the caller's
        plan.produce = true;                   // queries are something else the order is merely a poor one, never wrong
    }
    CU(cudaEventRecord(e->ev_sync, e->stream));
    CU(cudaStreamWaitEvent(l.stream, e->ev_sync, 0));
    CU(cudaMemcpyAsync(dq, records, (size_t)n * 32, cudaMemcpyHostToDevice, l.stream));
    if (dp) CU(cudaMemcpyAsync(dp, ply, (size_t)n * 4, cudaMemcpyHostToDevice, l.stream));
    if (dg) CU(cudaMemcpyAsync(dg, game_id, (size_t)n * 8, cudaMemcpyHostToDevice, l.stream));
    const SelectOut out = {nullptr, nullptr, nullptr, value ? (float *)dv : nullptr, n_seq ? (int32_t *)dn : nullptr, nullptr};
    AdvanceOut adv = {(int8_t *)dc, winner ? (int8_t *)dw : nullptr, (const int32_t *)dp, (const long long *)dg,
                      (uint32_t)dice_seed, (uint32_t)(dice_seed >> 32), nullptr, nullptr,
                      (long long)id_stride, first_mover, id_stride > 0 ? (int32_t *)dp : nullptr, id_stride > 0 ? (long long *)dg : nullptr};
    if ((rc = launch_select(e, l.stream, l.counter, l.steal, (const int8_t *)dq, n, epsilon, explore_seed, out, plan, e->lane_grid, adv))) return rc;
    if (plan.produce) { l.order_slot = 1 - plan.slot; l.order_n = n; }
    CU(cudaMemcpyAsync(next_records, dc, (size_t)n * 32, cudaMemcpyDeviceToHost, l.stream));
    if (winner) CU(cudaMemcpyAsync(winner, dw, (size_t)n, cudaMemcpyDeviceToHost, l.stream));
    if (value) CU(cudaMemcpyAsync(value, dv, (size_t)n * 4, cudaMemcpyDeviceToHost, l.stream));
    if (n_seq) CU(cudaMemcpyAsync(n_seq, dn, (size_t)n * 4, cudaMemcpyDeviceToHost, l.stream));
    if (id_stride > 0) {
        CU(cudaMemcpyAsync(ply, dp, (size_t)n * 4, cudaMemcpyDeviceToHost, l.stream));
        CU(cudaMemcpyAsync(game_id, dg, (size_t)n * 8, cudaMemcpyDeviceToHost, l.stream));
    }
    CU(cudaEventRecord(l.done, l.stream));
    l.busy = true;
    return BGX_OK;
}

// One iteration of play_game's loop (train.py:103-121) for n games through host buffers, asynchronous:
// make_move, is_game_over, setTurn, roll_dice.  = bgx_select_moves_host_async + bgx_advance_host in one queued call.
int bgx_play_ply_host_async(bgx_engine *e, int lane, const int8_t *records, const int32_t *next_ply, const int64_t *game_id,
                            int64_t n, float epsilon, uint64_t explore_seed, uint64_t dice_seed,
                            int8_t *next_records, int8_t *winner, float *value, int32_t *n_seq)
{
    USE(e);
    return play_ply(e, lane, records, const_cast<int32_t *>(next_ply), const_cast<int64_t *>(game_id), 0, 0, n, epsilon, explore_seed, dice_seed,
                    next_records, winner, value, n_seq, "bgx_play_ply_host_async");
}

// The same with the population's bookkeeping on the device: finished games restart in place, ply and game id travel with the records.
int bgx_play_ply_restart_host_async(bgx_engine *e, int lane, const int8_t *records, int32_t *ply, int64_t *game_id, int64_t id_stride,
                                    int first_mover, int64_t n, float epsilon, uint64_t explore_seed, uint64_t dice_seed,
                                    int8_t *next_records, int8_t *winner, float *value, int32_t *n_seq)
{
    USE(e);
    NEED(ply && game_id && id_stride > 0, "restart mode needs ply, game_id and a positive id_stride");
    NEED(first_mover == BGX_FIRST_ROLLOFF || first_mover == BGX_FIRST_PARITY, "unknown first-mover rule");
    return play_ply(e, lane, records, ply, game_id, id_stride, first_mover, n, epsilon, explore_seed, dice_seed,
                    next_records, winner, value, n_seq, "bgx_play_ply_restart_host_async");
}

int bgx_lane_wait(bgx_engine *e, int lane)
{
    USE(e);
    NEED(lane >= 0 && lane < kLanes, "lane out of range");
    bgx_lane &l = e->lanes[lane];
    if (!l.busy) return BGX_OK;
    CU(cudaEventSynchronize(l.done));
    l.busy = false;
    return BGX_OK;
}

int bgx_advance(bgx_engine *e, const int8_t *chosen, int8_t *next, int64_t n, uint64_t seed, int32_t ply,
                const int64_t *game_id, int8_t *winner)
{
    USE(e);
    NEED(chosen && next && n >= 0 && ply >= 0, "bad argument");
    if (n == 0) return BGX_OK;
    long long grid = (n + 7) / 8;
    if (grid > (long long)e->sm_count * 8) grid = (long long)e->sm_count * 8;
    k_advance<<<(int)grid, 256, 0, e->stream>>>(chosen, next, n, (uint32_t)seed, (uint32_t)(seed >> 32), ply,
                                                (const long long *)game_id, winner);
    e->launches++;
    CU(cudaGetLastError());
    return BGX_OK;
}

// ------------------------------------------------------------------------ self-play

static int ensure_td(bgx_engine *e);

int bgx_selfplay_init(bgx_engine *e, int64_t n_slots, int64_t first_id, int64_t id_stride, uint64_t seed,
                      int first_mover, int32_t traj_cap)
{
    USE(e);
    if (traj_cap > 0) {                              // a population that records trajectories will be replayed: allocate the replay's
        const int rc = ensure_td(e);                 // scratch now, not inside the first (timed) bgx_td_replay
        if (rc) return rc;
    }
    NEED(n_slots > 0 && id_stride > 0 && first_id >= 0 && traj_cap >= 0, "bad argument");
    NEED(first_mover == BGX_FIRST_ROLLOFF || first_mover == BGX_FIRST_PARITY, "unknown first-mover rule");
    CU(cudaStreamSynchronize(e->stream));
    cudaFree(e->slots); cudaFree(e->ply); cudaFree(e->game_id); cudaFree(e->traj_pre); cudaFree(e->traj_chosen);
    e->slots = nullptr; e->ply = nullptr; e->game_id = nullptr; e->traj_pre = nullptr; e->traj_chosen = nullptr;
    e->n_slots = 0;
    CU(cudaMalloc(&e->slots, (size_t)n_slots * 32));
    CU(cudaMalloc(&e->ply, (size_t)n_slots * 4));
    CU(cudaMalloc(&e->game_id, (size_t)n_slots * 8));
    if (traj_cap > 0) {
        CU(cudaMalloc(&e->traj_pre, (size_t)n_slots * traj_cap * 32));
        if (e->record_chosen) CU(cudaMalloc(&e->traj_chosen, (size_t)n_slots * traj_cap * 32));
    }
    e->n_slots = n_slots; e->first_id = first_id; e->id_stride = id_stride;
    e->seed_lo = (uint32_t)seed; e->seed_hi = (uint32_t)(seed >> 32);
    e->first_mover = first_mover; e->traj_cap = traj_cap;
    k_selfplay_reset<<<e->sm_count * 4, 256, 0, e->stream>>>(e->slots, e->ply, e->game_id, n_slots, first_id, id_stride, 0,
                                                            e->seed_lo, e->seed_hi, first_mover);
    e->launches++;
    CU(cudaGetLastError());
    return BGX_OK;
}

int bgx_selfplay_record_chosen(bgx_engine *e, int on)
{
    if (!e) { set_error("bgx_selfplay_record_chosen: null"); return BGX_E_INVALID; }
    e->record_chosen = on != 0;
    return BGX_OK;
}

int bgx_selfplay_next_round(bgx_engine *e)
{
    USE(e);
    if (e->n_slots == 0) { set_error("bgx_selfplay_next_round: call bgx_selfplay_init first"); return BGX_E_STATE; }
    k_selfplay_reset<<<e->sm_count * 4, 256, 0, e->stream>>>(e->slots, e->ply, e->game_id, e->n_slots, e->first_id, e->id_stride, 1,
                                                            e->seed_lo, e->seed_hi, e->first_mover);
    e->launches++;
    CU(cudaGetLastError());
    return BGX_OK;
}

static int run_selfplay(bgx_engine *e, int n_plies, int round_mode, float epsilon, bgx_stats *out)
{
    if (e->n_slots == 0) { set_error("self-play: call bgx_selfplay_init first"); return BGX_E_STATE; }
    if (!e->have_weights) { set_error("self-play: weights not set"); return BGX_E_STATE; }
    SelfplayParams p;
    p.slots = e->slots; p.ply = e->ply; p.game_id = e->game_id;
    p.traj_pre = e->traj_pre; p.traj_chosen = e->traj_chosen;
    p.n_slots = e->n_slots; p.id_stride = e->id_stride;
    p.seed_lo = e->seed_lo; p.seed_hi = e->seed_hi;
    p.first_mover = e->first_mover; p.traj_cap = e->traj_cap;
    p.n_plies = n_plies; p.round_mode = round_mode; p.epsilon = epsilon;
    p.counter = e->counter; p.stats = e->stats; p.zstash = e->zstash;
    CU(cudaMemsetAsync(e->counter, 0, sizeof(unsigned long long), e->stream));
    CU(cudaMemsetAsync(e->stats, 0, 16 * sizeof(unsigned long long), e->stream));
    tick(e);
#define BGX_LAUNCH_SELFPLAY(W, S, X) k_selfplay<W, S, X><<<game_grid(e), W * 32, ply_smem<W, S>(), e->stream>>>(p, e->fixed, e->flat, e->steal)
    const bool ex = epsilon > 0.f;
    if (e->selfplay_warps == 16) { if (ex) BGX_LAUNCH_SELFPLAY(16, 109, true); else BGX_LAUNCH_SELFPLAY(16, 109, false); }
    else if (e->selfplay_warps == 20) { if (ex) BGX_LAUNCH_SELFPLAY(20, 86, true); else BGX_LAUNCH_SELFPLAY(20, 86, false); }
    else if (e->selfplay_warps == 24) { if (ex) BGX_LAUNCH_SELFPLAY(24, 72, true); else BGX_LAUNCH_SELFPLAY(24, 72, false); }
    else { if (ex) BGX_LAUNCH_SELFPLAY(32, 53, true); else BGX_LAUNCH_SELFPLAY(32, 53, false); }
#undef BGX_LAUNCH_SELFPLAY
    tock(e);
    e->launches++;
    CU(cudaGetLastError());
    if (out) {
        unsigned long long h[8];
        CU(cudaMemcpyAsync(h, e->stats, sizeof h, cudaMemcpyDeviceToHost, e->stream));
        CU(cudaStreamSynchronize(e->stream));
        std::memset(out, 0, sizeof *out);
        out->plies = (int64_t)h[0]; out->sequences = (int64_t)h[1]; out->scored = (int64_t)h[2];
        out->games_finished = (int64_t)h[3]; out->p1_wins = (int64_t)h[4]; out->truncated = (int64_t)h[5];
        out->tree_edges = (int64_t)h[7];
    }
    return BGX_OK;
}

int bgx_selfplay_step(bgx_engine *e, int32_t n_plies, float epsilon, bgx_stats *out)
{
    USE(e);
    NEED(n_plies > 0, "n_plies must be positive");
    return run_selfplay(e, n_plies, 0, epsilon, out);
}

int bgx_selfplay_round(bgx_engine *e, float epsilon, bgx_stats *out)
{
    USE(e);
    return run_selfplay(e, 0, 1, epsilon, out);
}

int bgx_selfplay_read(bgx_engine *e, int8_t *records, int32_t *ply, int64_t *game_id)
{
    USE(e);
    if (e->n_slots == 0) { set_error("bgx_selfplay_read: call bgx_selfplay_init first"); return BGX_E_STATE; }
    if (records) CU(cudaMemcpyAsync(records, e->slots, (size_t)e->n_slots * 32, cudaMemcpyDeviceToHost, e->stream));
    if (ply) CU(cudaMemcpyAsync(ply, e->ply, (size_t)e->n_slots * 4, cudaMemcpyDeviceToHost, e->stream));
    if (game_id) CU(cudaMemcpyAsync(game_id, e->game_id, (size_t)e->n_slots * 8, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    return BGX_OK;
}

int bgx_export_trajectory(bgx_engine *e, int64_t slot, int32_t cap, int8_t *pre, int8_t *chosen, int32_t *T)
{
    USE(e);
    NEED(T && slot >= 0 && slot < e->n_slots, "bad slot");
    if (!e->traj_pre) { set_error("bgx_export_trajectory: population was created with traj_cap = 0"); return BGX_E_STATE; }
    int32_t ply = 0;
    CU(cudaMemcpyAsync(&ply, e->ply + slot, 4, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    if (ply > e->traj_cap) ply = e->traj_cap;
    *T = ply;
    if (ply > cap) { set_error("bgx_export_trajectory: %d plies, cap %d", ply, cap); return BGX_E_CAPACITY; }
    if (ply == 0) return BGX_OK;
    if (pre) CU(cudaMemcpyAsync(pre, e->traj_pre + (size_t)slot * e->traj_cap * 32, (size_t)ply * 32, cudaMemcpyDeviceToHost, e->stream));
    if (chosen) {
        if (!e->traj_chosen) { set_error("bgx_export_trajectory: chosen afterstates were not recorded (bgx_selfplay_record_chosen)"); return BGX_E_STATE; }
        CU(cudaMemcpyAsync(chosen, e->traj_chosen + (size_t)slot * e->traj_cap * 32, (size_t)ply * 32, cudaMemcpyDeviceToHost, e->stream));
    }
    CU(cudaStreamSynchronize(e->stream));
    return BGX_OK;
}

int bgx_selfplay_sample(bgx_engine *e, int32_t per_game, uint64_t seed, int8_t *records)
{
    USE(e);
    NEED(records && per_game > 0, "bad argument");
    if (e->n_slots == 0 || !e->traj_pre) { set_error("bgx_selfplay_sample: needs a population created with traj_cap > 0"); return BGX_E_STATE; }
    k_traj_sample<<<e->sm_count * 8, 256, 0, e->stream>>>(e->traj_pre, e->ply, e->n_slots, e->traj_cap, per_game,
                                                         (uint32_t)seed, (uint32_t)(seed >> 32), records);
    e->launches++;
    CU(cudaGetLastError());
    return BGX_OK;
}

int bgx_selfplay_sample_host(bgx_engine *e, int32_t per_game, uint64_t seed, int8_t *records)
{
    USE(e);
    NEED(records && per_game > 0, "bad argument");
    void *d;
    int rc;
    const size_t bytes = (size_t)e->n_slots * per_game * 32;
    if ((rc = scratch(e, 0, bytes, &d))) return rc;
    if ((rc = bgx_selfplay_sample(e, per_game, seed, (int8_t *)d))) return rc;
    CU(cudaMemcpyAsync(records, d, bytes, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    return BGX_OK;
}

// ------------------------------------------------------------------------ TD(lambda)

static int ensure_td(bgx_engine *e)
{
    if (e->td_partial) return BGX_OK;
    e->td_grid = e->sm_count * kTdCtasPerSm;
    CU(cudaMalloc(&e->td_partial, (size_t)e->td_grid * BGX_NPARAMS_PADDED * sizeof(float)));
    CU(cudaMalloc(&e->td_home, (size_t)e->td_grid * 2 * kTableBytes));
    CU(cudaMalloc(&e->td_delta, (size_t)BGX_NPARAMS_PADDED * sizeof(float)));
    CU(cudaMalloc(&e->td_prof, 128 * sizeof(unsigned long long)));
    CU(cudaMalloc(&e->td_sched, 2 * kTdSchedLen * sizeof(double)));
    return BGX_OK;
}

static int launch_td(bgx_engine *e, const int8_t *traj, const int8_t *slots, const int32_t *ply, long long n_games, int traj_cap,
                     double lr, double lambda, long long episode_first, float *delta_dev, float *final_weights, double *sq_errors, bgx_stats *out)
{
    int rc = ensure_td(e);
    if (rc) return rc;
    if (traj_cap > kTdMaxSteps) { set_error("TD replay: trajectories of up to %d recorded plies (traj_cap %d)", kTdMaxSteps, traj_cap); return BGX_E_INVALID; }
    int grid = e->td_grid;
    if (grid > n_games) grid = (int)n_games;
    TdParams p;
    p.traj = traj; p.slots = slots; p.ply = ply; p.n_games = n_games; p.traj_cap = traj_cap;
    p.lr = lr; p.lambda = (float)lambda;
    p.flat = e->flat; p.wt = e->wt; p.partial = e->td_partial;
    p.final_weights = final_weights; p.sq_errors = sq_errors;
    p.stats = e->stats; p.dstats = e->dstats;
    p.sched = nullptr; p.episode_first = 0;
    if (episode_first >= 0) {                        // the reference's schedule (model.py:69-73), tabulated with the host's libm pow
        double sched[2 * kTdSchedLen];
        for (int k = 0; k < kTdSchedLen; k++) {
            sched[k] = std::max(0.01, 0.1 * std::pow(0.96, (double)k));
            sched[kTdSchedLen + k] = std::max(0.7, 0.9 * std::pow(0.96, (double)k));
        }
        CU(cudaMemcpyAsync(e->td_sched, sched, sizeof sched, cudaMemcpyHostToDevice, e->stream));
        CU(cudaStreamSynchronize(e->stream));        // `sched` is on this stack frame
        p.sched = e->td_sched;
        p.episode_first = episode_first;
    }
    p.prof = e->td_prof;
    p.home = e->td_home;
    if (e->td_profile) CU(cudaMemsetAsync(e->td_prof, 0, 128 * sizeof(unsigned long long), e->stream));
    CU(cudaMemsetAsync(e->counter, 0, sizeof(unsigned long long), e->stream));
    CU(cudaMemsetAsync(e->stats, 0, 16 * sizeof(unsigned long long), e->stream));
    CU(cudaMemsetAsync(e->dstats, 0, 2 * sizeof(double), e->stream));
    tick(e);
    if (e->td_profile) k_td_replay<true><<<grid, kTdThreads, kTdSmem, e->stream>>>(p);
    else k_td_replay<false><<<grid, kTdThreads, kTdSmem, e->stream>>>(p);
    e->launches++;
    CU(cudaGetLastError());
    if (delta_dev) {
        k_td_reduce<<<(BGX_NPARAMS_PADDED + 255) / 256, 256, 0, e->stream>>>(e->td_partial, grid, delta_dev);
        e->launches++;
        CU(cudaGetLastError());
    }
    tock(e);
    if (out) {
        unsigned long long h[16];
        double d[2];
        CU(cudaMemcpyAsync(h, e->stats, sizeof h, cudaMemcpyDeviceToHost, e->stream));
        CU(cudaMemcpyAsync(d, e->dstats, sizeof d, cudaMemcpyDeviceToHost, e->stream));
        CU(cudaStreamSynchronize(e->stream));
        std::memset(out, 0, sizeof *out);
        out->td_steps = (int64_t)h[6];
        out->games_finished = (int64_t)h[3];
        out->truncated = (int64_t)h[5];
        out->td_sq_error = d[0];
        out->td_lazy_row_steps = (int64_t)h[7];
        out->td_live_rows = (int64_t)h[8];
    }
    return BGX_OK;
}

static int td_replay_population(bgx_engine *e, double lr, double lambda, long long episode_first, float *delta_dev, bgx_stats *out)
{
    NEED(delta_dev, "null delta buffer");
    if (e->n_slots == 0 || !e->traj_pre) { set_error("TD replay: needs a population created with traj_cap > 0"); return BGX_E_STATE; }
    if (!e->have_weights) { set_error("TD replay: weights not set"); return BGX_E_STATE; }
    return launch_td(e, e->traj_pre, e->slots, e->ply, e->n_slots, e->traj_cap, lr, lambda, episode_first, delta_dev, nullptr, nullptr, out);
}

int bgx_td_replay(bgx_engine *e, double lr, double lambda, float *delta_dev, bgx_stats *out)
{
    USE(e);
    return td_replay_population(e, lr, lambda, -1, delta_dev, out);
}

int bgx_td_replay_scheduled(bgx_engine *e, int64_t games_done, float *delta_dev, bgx_stats *out)
{
    USE(e);
    NEED(games_done >= 0, "games_done must not be negative");
    return td_replay_population(e, 0.0, 0.0, (long long)games_done + e->first_id + 1, delta_dev, out);
}

int bgx_apply_delta(bgx_engine *e, const float *delta_dev, float scale)
{
    USE(e);
    NEED(delta_dev, "null delta buffer");
    if (int rc = lanes_idle(e, "bgx_apply_delta")) return rc;
    k_axpy<<<(BGX_NPARAMS + 255) / 256, 256, 0, e->stream>>>(e->flat, delta_dev, scale, BGX_NPARAMS);
    e->launches++;
    CU(cudaGetLastError());
    return rebuild_table(e);
}

// bgx_td_replay + bgx_apply_delta for a single-GPU caller without device buffers of its own (the pybind11 module)
int bgx_td_round_host(bgx_engine *e, double lr, double lambda, float scale, float *delta_host, bgx_stats *out)
{
    USE(e);
    int rc = ensure_td(e);
    if (rc) return rc;
    float *dd = e->td_delta;
    if ((rc = bgx_td_replay(e, lr, lambda, dd, out))) return rc;
    if (delta_host) {
        CU(cudaMemcpyAsync(delta_host, dd, (size_t)BGX_NPARAMS * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
        CU(cudaStreamSynchronize(e->stream));
    }
    return scale != 0.f ? bgx_apply_delta(e, dd, scale) : BGX_OK;
}

int bgx_td_replay_host(bgx_engine *e, const int8_t *records, int32_t T, int player1_won, double lr, double lambda,
                       float *new_W1, float *new_b1, float *new_w2, float *new_b2, double *sq_errors)
{
    USE(e);
    NEED(records && T > 0 && T <= kTdMaxSteps && new_W1 && new_b1 && new_w2 && new_b2, "bad argument (1 <= T <= BGX_TD_MAX_STEPS)");
    if (!e->have_weights) { set_error("bgx_td_replay_host: weights not set"); return BGX_E_STATE; }
    void *dtraj, *dslot, *dply, *dfinal, *dsq;
    int rc;
    if ((rc = scratch(e, 0, (size_t)T * 32, &dtraj))) return rc;
    if ((rc = scratch(e, 1, 32, &dslot))) return rc;
    if ((rc = scratch(e, 2, 4, &dply))) return rc;
    if ((rc = scratch(e, 9, BGX_NPARAMS_PADDED * sizeof(float), &dfinal))) return rc;
    if ((rc = scratch(e, 10, (size_t)T * 8, &dsq))) return rc;
    int8_t slot[32] = {0};
    slot[31] = player1_won ? kP1Won : kP2Won;
    CU(cudaMemcpyAsync(dtraj, records, (size_t)T * 32, cudaMemcpyHostToDevice, e->stream));
    CU(cudaMemcpyAsync(dslot, slot, 32, cudaMemcpyHostToDevice, e->stream));
    CU(cudaMemcpyAsync(dply, &T, 4, cudaMemcpyHostToDevice, e->stream));
    CU(cudaMemsetAsync(dsq, 0, (size_t)T * 8, e->stream));
    if ((rc = launch_td(e, (const int8_t *)dtraj, (const int8_t *)dslot, (const int32_t *)dply, 1, T, lr, lambda, -1,
                        nullptr, (float *)dfinal, (double *)dsq, nullptr)))
        return rc;
    std::vector<float> flat(BGX_NPARAMS_PADDED);
    CU(cudaMemcpyAsync(flat.data(), dfinal, flat.size() * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
    if (sq_errors && T > 1) CU(cudaMemcpyAsync(sq_errors, dsq, (size_t)(T - 1) * 8, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    std::memcpy(new_W1, flat.data(), kTableFloats * sizeof(float));
    std::memcpy(new_b1, flat.data() + kTableFloats, kHidden * sizeof(float));
    std::memcpy(new_w2, flat.data() + kTableFloats + kHidden, kHidden * sizeof(float));
    new_b2[0] = flat[kTableFloats + 2 * kHidden];
    return BGX_OK;
}

// ------------------------------------------------------------------------ the cross-GPU exchange (SURVEY 8e)
// NCCL is bound at run time (dlopen), so that libbgx has no link-time dependency on it and single-GPU users need none.
namespace {
struct NcclUniqueId { char internal[128]; };
struct NcclApi {
    void *lib = nullptr;
    int (*GetUniqueId)(NcclUniqueId *) = nullptr;
    int (*CommInitRank)(void **, int, NcclUniqueId, int) = nullptr;
    int (*CommDestroy)(void *) = nullptr;
    int (*AllReduce)(const void *, void *, size_t, int, int, void *, cudaStream_t) = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
};
NcclApi g_nccl;

int nccl_load(const char *path)
{
    if (g_nccl.AllReduce) return BGX_OK;
    void *lib = nullptr;
    const char *tried[] = {path, "libnccl.so.2", "libnccl.so"};
    for (const char *name : tried)
        if (name && *name && (lib = dlopen(name, RTLD_NOW | RTLD_GLOBAL))) break;
    if (!lib) { set_error("NCCL: cannot load libnccl (%s)", dlerror()); return BGX_E_STATE; }
    g_nccl.GetUniqueId = (int (*)(NcclUniqueId *))dlsym(lib, "ncclGetUniqueId");
    g_nccl.CommInitRank = (int (*)(void **, int, NcclUniqueId, int))dlsym(lib, "ncclCommInitRank");
    g_nccl.CommDestroy = (int (*)(void *))dlsym(lib, "ncclCommDestroy");
    g_nccl.AllReduce = (int (*)(const void *, void *, size_t, int, int, void *, cudaStream_t))dlsym(lib, "ncclAllReduce");
    g_nccl.GetErrorString = (const char *(*)(int))dlsym(lib, "ncclGetErrorString");
    if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.CommDestroy || !g_nccl.AllReduce) {
        g_nccl = NcclApi();
        set_error("NCCL: libnccl lacks an expected symbol");
        return BGX_E_STATE;
    }
    g_nccl.lib = lib;
    return BGX_OK;
}
int nccl_check(int rc, const char *what)
{
    if (rc == 0) return BGX_OK;
    set_error("NCCL: %s failed: %s", what, g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "?");
    return BGX_E_CUDA;
}
} // namespace

int bgx_nccl_load(const char *libnccl_path) { return nccl_load(libnccl_path); }

int bgx_nccl_unique_id(void *id128)
{
    NEED(id128, "null id buffer");
    int rc = nccl_load(nullptr);
    if (rc) return rc;
    return nccl_check(g_nccl.GetUniqueId((NcclUniqueId *)id128), "ncclGetUniqueId");
}

int bgx_nccl_comm_init(bgx_engine *e, int n_ranks, int rank, const void *id128, void **comm)
{
    USE(e);
    NEED(id128 && comm && n_ranks > 0 && rank >= 0 && rank < n_ranks, "bad argument");
    int rc = nccl_load(nullptr);
    if (rc) return rc;
    NcclUniqueId id;
    std::memcpy(&id, id128, sizeof id);
    return nccl_check(g_nccl.CommInitRank(comm, n_ranks, id, rank), "ncclCommInitRank");
}

int bgx_nccl_comm_destroy(void *comm)
{
    if (!comm) return BGX_OK;
    int rc = nccl_load(nullptr);
    if (rc) return rc;
    return nccl_check(g_nccl.CommDestroy(comm), "ncclCommDestroy");
}

// the only cross-GPU traffic of the path: sum of the per-rank weight deltas, fp32[25,604], in place, on the engine's stream
int bgx_allreduce_delta(bgx_engine *e, void *nccl_comm, float *delta_dev)
{
    USE(e);
    NEED(nccl_comm && delta_dev, "null communicator or buffer");
    int rc = nccl_load(nullptr);
    if (rc) return rc;
    return nccl_check(g_nccl.AllReduce(delta_dev, delta_dev, BGX_NPARAMS_PADDED, /*ncclFloat32*/ 7, /*ncclSum*/ 0, nccl_comm, e->stream), "ncclAllReduce");
}

// ------------------------------------------------------------------------ introspection

int bgx_td_profile(bgx_engine *e, int on, uint64_t *cycles)
{
    USE(e);
    int rc = ensure_td(e);
    if (rc) return rc;
    e->td_profile = on != 0;
    if (cycles) {
        CU(cudaStreamSynchronize(e->stream));
        CU(cudaMemcpy(cycles, e->td_prof, 128 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    }
    return BGX_OK;
}

int bgx_launch_count(bgx_engine *e, int64_t *n)
{
    if (!e || !n) { set_error("bgx_launch_count: null"); return BGX_E_INVALID; }
    *n = e->launches;
    return BGX_OK;
}

int bgx_last_kernel_ms(bgx_engine *e, float *ms)
{
    USE(e);
    NEED(ms, "null");
    if (!e->timed) { set_error("bgx_last_kernel_ms: nothing launched yet"); return BGX_E_STATE; }
    CU(cudaEventSynchronize(e->ev1));
    CU(cudaEventElapsedTime(ms, e->ev0, e->ev1));
    return BGX_OK;
}

int bgx_sfu_monotone(bgx_engine *e, int64_t *ex2_violations, int64_t *rcp_violations)
{
    USE(e);
    NEED(ex2_violations && rcp_violations, "null");
    CU(cudaMemsetAsync(e->stats, 0, 16 * sizeof(unsigned long long), e->stream));
    k_sfu_monotone<<<e->sm_count * 8, 256, 0, e->stream>>>(e->stats);
    e->launches++;
    CU(cudaGetLastError());
    unsigned long long h[2];
    CU(cudaMemcpyAsync(h, e->stats, sizeof h, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    *ex2_violations = (int64_t)h[0];
    *rcp_violations = (int64_t)h[1];
    return BGX_OK;
}

int bgx_kernel_config(bgx_engine *e, int *selfplay_warps, int *select_warps)
{
    if (!e) { set_error("bgx_kernel_config: null"); return BGX_E_INVALID; }
    if (selfplay_warps) *selfplay_warps = e->selfplay_warps;
    if (select_warps) *select_warps = e->select_warps;
    return BGX_OK;
}

int bgx_device_props(bgx_engine *e, int *sm_count, int *clock_khz, int64_t *global_mem)
{
    if (!e) { set_error("bgx_device_props: null"); return BGX_E_INVALID; }
    if (sm_count) *sm_count = e->sm_count;
    if (clock_khz) *clock_khz = e->clock_khz;
    if (global_mem) *global_mem = (int64_t)e->global_mem;
    return BGX_OK;
}

} // extern "C"
