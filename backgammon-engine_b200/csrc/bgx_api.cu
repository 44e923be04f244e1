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
#include <type_traits>
#include <vector>

using namespace bgx;

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

// device buffers that are kept from call to call and grow on demand
template <int K>
struct Arena {
    void *buf[K] = {};
    size_t cap[K] = {};

    // buffer i with room for `bytes`; a buffer too small is freed and reallocated with headroom, its contents lost
    template <typename T>
    int grow(int i, size_t bytes, T **out)
    {
        if (cap[i] < bytes) {
            if (buf[i]) CU(cudaFree(buf[i]));
            buf[i] = nullptr;
            cap[i] = 0;
            const size_t want = bytes + bytes / 4 + 256;
            CU(cudaMalloc(&buf[i], want));
            cap[i] = want;
        }
        *out = static_cast<T *>(buf[i]);
        return BGX_OK;
    }
    void release() { for (void *b : buf) cudaFree(b); }
};

// the work buffers of the device-form entry points, by name
enum Work {
    kSelectOrder,                                    // bgx_select_moves: sorted queue
    kEnumScanSums,                                   // bgx_enumerate_count: tile sums of the scan
    // bgx_select_moves_2ply, per query: summary walk, candidate counts and offsets, expansion counts and offsets
    kTpSeq, kTpUnique, kTpDigest, kTpCount, kTpOffsets, kTpScanSums, kTpFlags, kTpExpandCount, kTpExpandOffsets,
    // per candidate: record, first sequence, one-ply value, expanded?, two-ply value; the list of expanded candidates
    kTpRecords, kTpMoves, kTpMovesLen, kTpValue, kTpExpand, kTpE2, kTpList,
    // per chunk of replies: records, values, sorted queue
    kTpReplies, kTpReplyValue, kTpReplyOrder,
    // bgx_rollout / bgx_rollout_vr: the per-trial results of a chunk the caller did not ask for
    kRolloutValue, kRolloutOutcome, kRolloutPlies, kRolloutLuck,
    kRolloutRolls, kRolloutZlist,                    // k_rollout_vr: per warp, the roll values of its ply and the 21-roll walks' stash
    kWorkBufs
};
enum LaneWork { kLaneOrder0, kLaneOrder1, kLaneWorkBufs };   // a lane's sorted queues: the one read, the one written for the next call
constexpr int kStageBufs = 10;                   // the most host arrays one *_host call stages (bgx_rollout_vr_host)

// an asynchronous lane of the batched make_move path: its own stream, work-queue counter,
// sharing buffer and staging buffers, so that two batches can be in flight at once
struct bgx_lane {
    cudaStream_t stream = nullptr;
    cudaEvent_t done = nullptr;
    unsigned long long *counter = nullptr;   // [0] work queue, [8..15] the 16 bucket totals of k_select_order
    StealResult *steal = nullptr;
    Arena<kLaneWorkBufs> work;
    Arena<kStageBufs> stage;
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
    Arena<kWorkBufs> work;                   // buffers of the device-form calls (enum Work)
    Arena<kStageBufs> stage;                 // device copies of the host arrays of the *_host calls (Stage)
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

// The host side of a *_host call on the engine's stream or on a lane's.  in() and out() hand out staging buffers in call
// order from an arena that no device-form call touches, so that they can never alias the buffers of the call they wrap.
// The first failing CUDA call leaves its message in bgx_last_error and its code in rc; later ones are skipped.
struct Stage {
    Arena<kStageBufs> &arena;
    cudaStream_t stream;
    bgx_lane *lane;                          // null: the engine's stream
    int rc = BGX_OK, used = 0, n_back = 0;
    struct Back { void *host; const void *dev; size_t bytes; } back[kStageBufs];

    explicit Stage(bgx_engine *e) : arena(e->stage), stream(e->stream), lane(nullptr) {}
    explicit Stage(bgx_lane &l) : arena(l.stage), stream(l.stream), lane(&l) {}

    template <typename T>
    T *take(size_t bytes)
    {
        T *d = nullptr;
        if (rc == BGX_OK && used == kStageBufs) { set_error("staging: more than %d buffers", kStageBufs); rc = BGX_E_STATE; }
        if (rc == BGX_OK) rc = arena.grow(used++, bytes, &d);
        return d;
    }
    int h2d(void *dev, const void *host, size_t bytes) { CU(cudaMemcpyAsync(dev, host, bytes, cudaMemcpyHostToDevice, stream)); return BGX_OK; }
    // a device copy of `host` (null for a null host pointer)
    template <typename T>
    T *in(const T *host, size_t bytes)
    {
        if (!host) return nullptr;
        T *d = take<T>(bytes);
        if (rc == BGX_OK) rc = h2d(d, host, bytes);
        return d;
    }
    // a device buffer whose contents finish() copies to `host` (null for a null host pointer: the call skips that output)
    template <typename T>
    T *out(T *host, size_t bytes)
    {
        if (!host) return nullptr;
        T *d = take<T>(bytes);
        copy_back(host, d, bytes);
        return d;
    }
    void copy_back(void *host, const void *dev, size_t bytes) { back[n_back++] = {host, dev, bytes}; }
    // after the device call (its return code is passed through): the copies back, then the stream synchronised, or the
    // lane marked busy until they are done
    int finish(int call_rc = BGX_OK)
    {
        if (call_rc != BGX_OK) return call_rc;
        for (int i = 0; i < n_back; i++) CU(cudaMemcpyAsync(back[i].host, back[i].dev, back[i].bytes, cudaMemcpyDeviceToHost, stream));
        n_back = 0;
        if (!lane) CU(cudaStreamSynchronize(stream));
        else {
            CU(cudaEventRecord(lane->done, stream));
            lane->busy = true;
        }
        return BGX_OK;
    }
};

static int need_weights(bgx_engine *e, const char *who)
{
    if (!e->have_weights) { set_error("%s: weights not set", who); return BGX_E_STATE; }
    return BGX_OK;
}

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

static int tick_(bgx_engine *e) { CU(cudaEventRecord(e->ev0, e->stream)); return BGX_OK; }
static int tock_(bgx_engine *e) { CU(cudaEventRecord(e->ev1, e->stream)); e->timed = true; return BGX_OK; }
#define tick(e) do { const int rc__ = tick_(e); if (rc__ != BGX_OK) return rc__; } while (0)
#define tock(e) do { const int rc__ = tock_(e); if (rc__ != BGX_OK) return rc__; } while (0)

static int game_grid(bgx_engine *e) { return e->sm_count; }   // persistent: one 16-warp CTA per SM

// f(std::true_type) or f(std::false_type): the kExplore instantiation of a fused ply kernel
template <typename F>
static void dispatch_explore(bool explore, F &&f)
{
    if (explore) f(std::true_type{});
    else f(std::false_type{});
}

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
    static_assert(PlyConfigs::fits(232448), "fused ply kernels: shared memory per CTA");
    const int rc = PlyConfigs::each([](auto c) {
        constexpr int W = decltype(c)::kWarps, S = decltype(c)::kSets;
        CU(cudaFuncSetAttribute(k_select<W, S, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, c.kSmem));
        CU(cudaFuncSetAttribute(k_select<W, S, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, c.kSmem));
        CU(cudaFuncSetAttribute(k_selfplay<W, S, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, c.kSmem));
        CU(cudaFuncSetAttribute(k_selfplay<W, S, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, c.kSmem));
        CU(cudaFuncSetAttribute(k_rollout<W, S>, cudaFuncAttributeMaxDynamicSharedMemorySize, c.kSmem));
        CU(cudaFuncSetAttribute(k_rollout_vr<W, S>, cudaFuncAttributeMaxDynamicSharedMemorySize, c.kSmem));
        return BGX_OK;
    });
    if (rc) return rc;
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
//   "rollout_warps"                    warps per CTA of k_rollout and k_rollout_vr: 16, 20, 24 or 32
//   "rollout_chunk"                    trials (games) per k_rollout launch, rounded down to whole positions (0: 2^24)
int bgx_set_option(bgx_engine *e, const char *key, int64_t value)
{
    if (!e || !key) { set_error("bgx_set_option: null"); return BGX_E_INVALID; }
    const std::string k(key);
    if (k == "selfplay_warps" || k == "select_warps" || k == "rollout_warps") {
        if (!PlyConfigs::has(value)) { set_error("bgx_set_option: %s must be 16, 20, 24 or 32", key); return BGX_E_INVALID; }
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
    e->work.release();
    e->stage.release();
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
        l.work.release();
        l.stage.release();
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

// the flat weight layout [W1[128][198] | b1[128] | w2[128] | b2[1]] and the state_dict tensors
static void pack_weights(float *flat, const float *W1, const float *b1, const float *w2, const float *b2)
{
    std::memcpy(flat, W1, kTableFloats * sizeof(float));
    std::memcpy(flat + kTableFloats, b1, kHidden * sizeof(float));
    std::memcpy(flat + kTableFloats + kHidden, w2, kHidden * sizeof(float));
    flat[kTableFloats + 2 * kHidden] = b2[0];
}
static void unpack_weights(const float *flat, float *W1, float *b1, float *w2, float *b2)
{
    std::memcpy(W1, flat, kTableFloats * sizeof(float));
    std::memcpy(b1, flat + kTableFloats, kHidden * sizeof(float));
    std::memcpy(w2, flat + kTableFloats + kHidden, kHidden * sizeof(float));
    b2[0] = flat[kTableFloats + 2 * kHidden];
}

int bgx_set_weights(bgx_engine *e, const float *W1, const float *b1, const float *w2, const float *b2)
{
    USE(e);
    NEED(W1 && b1 && w2 && b2, "null weight pointer");
    if (int rc = lanes_idle(e, "bgx_set_weights")) return rc;
    std::vector<float> flat(BGX_NPARAMS_PADDED, 0.f);
    pack_weights(flat.data(), W1, b1, w2, b2);
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
    unpack_weights(flat.data(), W1, b1, w2, b2);
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
    Stage s(e);
    const int8_t *dq = s.in(queries, (size_t)n * 32);
    int32_t *dn = s.out(n_seq, (size_t)n * 4);
    int32_t *du = s.out(n_unique, (size_t)n * 4);
    uint64_t *dd = s.out(digest, (size_t)n * 8);
    if (s.rc) return s.rc;
    return s.finish(bgx_enumerate_summary(e, dq, n, dn, du, dd));
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

// exclusive prefix sum of cnt[n] into offsets[n + 1]: three launches
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

// sizes of every query's sequence list and their exclusive prefix sum, on the device: the allocation pass of the
// materialised enumeration (a count-only walk, no dedup table, no digest) + the scan
int bgx_enumerate_count(bgx_engine *e, const int8_t *queries, int64_t n, int32_t *n_seq, int64_t *offsets)
{
    USE(e);
    NEED(queries && n_seq && offsets && n >= 0, "bad argument");
    if (n == 0) { CU(cudaMemsetAsync(offsets, 0, 8, e->stream)); return BGX_OK; }
    const int n_tiles = (int)((n + kScanTile - 1) / kScanTile);
    long long *sums;
    if (int rc = e->work.grow(kEnumScanSums, (size_t)(n_tiles + 1) * 8, &sums)) return rc;
    CU(cudaMemsetAsync(e->counter, 0, sizeof(unsigned long long), e->stream));
    tick(e);
    k_enumerate_count<<<e->sm_count * 2, kGameThreads, 0, e->stream>>>(queries, n, n_seq, e->counter);
    tock(e);
    e->launches++;
    return scan_counts(e, n_seq, n, (long long *)offsets, sums);
}

int bgx_enumerate_host(bgx_engine *e, const int8_t *queries, int64_t n, int64_t cap, int64_t *offsets,
                       int8_t *seq_moves, int8_t *seq_len, int8_t *states, int64_t *total)
{
    USE(e);
    NEED(queries && total && n >= 0 && cap >= 0, "bad argument");
    *total = 0;
    if (n == 0) { if (offsets) offsets[0] = 0; return BGX_OK; }
    Stage s(e);
    const int8_t *dq = s.in(queries, (size_t)n * 32);
    int32_t *dn = s.take<int32_t>((size_t)n * 4);
    int64_t *doff = s.take<int64_t>((size_t)(n + 1) * 8);
    if (s.rc) return s.rc;
    // the one number the host needs before it can size anything: 8 bytes
    int64_t rows_needed = 0;
    s.copy_back(&rows_needed, doff + n, 8);
    if (offsets) s.copy_back(offsets, doff, (size_t)(n + 1) * 8);
    if (int rc = s.finish(bgx_enumerate_count(e, dq, n, dn, doff))) return rc;
    *total = rows_needed;
    if (rows_needed > cap) { set_error("bgx_enumerate_host: %lld rows needed, cap %lld", (long long)rows_needed, (long long)cap); return BGX_E_CAPACITY; }
    NEED(seq_moves && seq_len && states, "null output buffer");
    const size_t rows = (size_t)rows_needed;
    if (rows == 0) return BGX_OK;
    int8_t *dm = s.out(seq_moves, rows * 8);
    int8_t *dl = s.out(seq_len, rows);
    int8_t *ds = s.out(states, rows * 32);
    if (s.rc) return s.rc;
    return s.finish(bgx_enumerate(e, dq, n, doff, dm, dl, ds));
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
    Stage s(e);
    const int8_t *dq = s.in(records, (size_t)n * 32);
    float *dx = s.out(X, (size_t)n * kFeatures * 4);
    if (s.rc) return s.rc;
    return s.finish(bgx_encode(e, dq, n, dx));
}

int bgx_evaluate(bgx_engine *e, const int8_t *records, int64_t n, float *V)
{
    USE(e);
    NEED(records && V && n >= 0, "bad argument");
    if (int rc = need_weights(e, "bgx_evaluate")) return rc;
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
    Stage s(e);
    const int8_t *dq = s.in(records, (size_t)n * 32);
    float *dv = s.out(V, (size_t)n * 4);
    if (s.rc) return s.rc;
    return s.finish(bgx_evaluate(e, dq, n, dv));
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
    PlyConfigs::dispatch(e->select_warps, [&](auto c) {
        constexpr int W = decltype(c)::kWarps, S = decltype(c)::kSets;
        dispatch_explore(epsilon > 0.f, [&](auto x) {
            k_select<W, S, decltype(x)::value><<<grid, W * 32, ply_smem<W, S>(), stream>>>(
                queries, n, epsilon, (uint32_t)seed, (uint32_t)(seed >> 32), out, e->fixed, e->flat, counter, steal, tune, region, totals, adv);
        });
    });
    e->launches++;
    CU(cudaGetLastError());
    return BGX_OK;
}

int bgx_select_moves(bgx_engine *e, const int8_t *queries, int64_t n, float epsilon, uint64_t seed,
                     int8_t *chosen, int8_t *moves, int8_t *moves_len, float *value, int32_t *n_seq, int32_t *n_scored)
{
    USE(e);
    NEED(queries && n >= 0, "bad argument");
    if (int rc = need_weights(e, "bgx_select_moves")) return rc;
    if (n == 0) return BGX_OK;
    const SelectOut out = {chosen, moves, moves_len, value, n_seq, n_scored};
    OrderPlan plan;
    if (n <= e->select_order_max) {
        if (int rc = e->work.grow(kSelectOrder, (size_t)n * kOrderBuckets * 4, &plan.region[0])) return rc;
    }
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
    Stage s(e);
    const int8_t *dq = s.in(queries, (size_t)n * 32);
    int8_t *dc = s.out(chosen, (size_t)n * 32);
    int8_t *dm = s.out(moves, (size_t)n * 8);
    int8_t *dl = s.out(moves_len, (size_t)n);
    float *dv = s.out(value, (size_t)n * 4);
    int32_t *dn = s.out(n_seq, (size_t)n * 4);
    int32_t *ds = s.out(n_scored, (size_t)n * 4);
    if (s.rc) return s.rc;
    return s.finish(bgx_select_moves(e, dq, n, epsilon, seed, dc, dm, dl, dv, dn, ds));
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

int bgx_select_moves_2ply(bgx_engine *e, const int8_t *queries, int64_t n, int32_t max_candidates,
                          int8_t *chosen, int8_t *moves, int8_t *moves_len, float *value, int32_t *n_candidates, int32_t *n_expanded)
{
    USE(e);
    NEED(queries && n >= 0 && max_candidates >= 0, "bad argument");
    if (int rc = need_weights(e, "bgx_select_moves_2ply")) return rc;
    if (n == 0) return BGX_OK;
    int rc = ensure_uniq_tables(e);
    if (rc) return rc;
    if (e->twoply_timing) {
        if (!e->tp0) { CU(cudaEventCreate(&e->tp0)); CU(cudaEventCreate(&e->tp1)); }
        CU(cudaEventRecord(e->tp0, e->stream));
    }
    const int n_tiles = (int)((n + kScanTile - 1) / kScanTile);
    int32_t *nseq, *uniq, *cnt, *nexp;
    unsigned long long *dig;
    long long *off, *eoff, *sums;
    int *flags;
    if ((rc = e->work.grow(kTpSeq, (size_t)n * 4, &nseq))) return rc;
    if ((rc = e->work.grow(kTpUnique, (size_t)n * 4, &uniq))) return rc;
    if ((rc = e->work.grow(kTpDigest, (size_t)n * 8, &dig))) return rc;
    if ((rc = e->work.grow(kTpCount, (size_t)n * 4, &cnt))) return rc;
    if ((rc = e->work.grow(kTpOffsets, (size_t)(n + 1) * 8, &off))) return rc;
    if ((rc = e->work.grow(kTpScanSums, (size_t)(n_tiles + 1) * 8, &sums))) return rc;
    if ((rc = e->work.grow(kTpFlags, 16, &flags))) return rc;
    if ((rc = e->work.grow(kTpExpandCount, (size_t)n * 4, &nexp))) return rc;
    if ((rc = e->work.grow(kTpExpandOffsets, (size_t)(n + 1) * 8, &eoff))) return rc;

    // 1. candidates: U per query (the summary walk), their offsets, then every distinct afterstate with its first sequence and V
    CU(cudaMemsetAsync(flags, 0, 16, e->stream));
    CU(cudaMemsetAsync(e->counter, 0, sizeof(unsigned long long), e->stream));
    k_enumerate_summary<<<e->uniq_grid, kGameThreads, 0, e->stream>>>(queries, n, nseq, uniq, dig, e->uniq_tables, e->uniq_gens, e->counter);
    k_twoply_count<<<(unsigned)((n + 255) / 256), 256, 0, e->stream>>>(uniq, n, cnt, flags);
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
    int8_t *rec, *cmv, *clen, *expand;
    float *val, *e2;
    const size_t C = (size_t)(n_cand > 0 ? n_cand : 1);
    if ((rc = e->work.grow(kTpRecords, C * 32, &rec))) return rc;
    if ((rc = e->work.grow(kTpMoves, C * 8, &cmv))) return rc;
    if ((rc = e->work.grow(kTpMovesLen, C, &clen))) return rc;
    if ((rc = e->work.grow(kTpValue, C * 4, &val))) return rc;
    if ((rc = e->work.grow(kTpExpand, C, &expand))) return rc;
    if ((rc = e->work.grow(kTpE2, C * 4, &e2))) return rc;
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
    long long *list;
    if ((rc = e->work.grow(kTpList, (size_t)(n_exp > 0 ? n_exp : 1) * 8, &list))) return rc;
    if (n_exp > 0) {
        k_twoply_list<<<small_grid, 256, 0, e->stream>>>(n, cnt, off, expand, eoff, list);
        e->launches++;
    }
    TWOPLY_MARK(e, 1);

    // 3. replies in chunks: 21 records per expanded candidate, k_select (values only), the expectation
    const long long chunk_replies = std::max<long long>(e->twoply_chunk > 0 ? e->twoply_chunk : kTwoplyChunk, kRolls);
    const long long per_chunk = chunk_replies / kRolls;
    const long long cap_replies = std::min<long long>(n_exp, per_chunk) * kRolls;
    int8_t *rep = nullptr;
    float *rval = nullptr;
    int32_t *region = nullptr;
    if (n_exp > 0) {
        if ((rc = e->work.grow(kTpReplies, (size_t)cap_replies * 32, &rep))) return rc;
        if ((rc = e->work.grow(kTpReplyValue, (size_t)cap_replies * 4, &rval))) return rc;
        if (cap_replies <= e->select_order_max && (rc = e->work.grow(kTpReplyOrder, (size_t)cap_replies * kOrderBuckets * 4, &region))) return rc;
    }
    for (long long e0 = 0; e0 < n_exp; e0 += per_chunk) {
        const long long e1 = std::min(n_exp, e0 + per_chunk);
        const long long nr = (e1 - e0) * kRolls;
        k_twoply_replies<<<(unsigned)std::min<long long>((nr + 7) / 8, (long long)e->sm_count * 16), 256, 0, e->stream>>>(list, e0, nr, rec, rep);
        e->launches++;
        const SelectOut out = {nullptr, nullptr, nullptr, rval, nullptr, nullptr};
        OrderPlan plan;
        plan.region[0] = nr <= e->select_order_max ? region : nullptr;
        if ((rc = launch_select(e, e->stream, e->counter, e->steal, rep, nr, 0.f, 0, out, plan))) return rc;
        TWOPLY_MARK(e, 2);
        k_twoply_reduce<<<game_grid(e), kGameThreads, kEvalSmem, e->stream>>>(list, e0, e1, rec, rval, e2, e->fixed);
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
    if (int rc = need_weights(e, "bgx_select_moves_2ply_host")) return rc;
    if (n == 0) return BGX_OK;
    Stage s(e);
    const int8_t *dq = s.in(queries, (size_t)n * 32);
    int8_t *dc = s.out(chosen, (size_t)n * 32);
    int8_t *dm = s.out(moves, (size_t)n * 8);
    int8_t *dl = s.out(moves_len, (size_t)n);
    float *dv = s.out(value, (size_t)n * 4);
    int32_t *dn = s.out(n_candidates, (size_t)n * 4);
    int32_t *dx = s.out(n_expanded, (size_t)n * 4);
    if (s.rc) return s.rc;
    return s.finish(bgx_select_moves_2ply(e, dq, n, max_candidates, dc, dm, dl, dv, dn, dx));
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

// bgx_rollout (vr_plies < 0: k_rollout) and bgx_rollout_vr (k_rollout_vr), arguments checked
static int rollout_run(bgx_engine *e, const int8_t *positions, int64_t n, int32_t trials, int32_t max_plies, uint64_t seed, int flags,
                       int32_t vr_plies, double *mean, double *std_err, int64_t *counts, float *trial_value, int8_t *trial_outcome,
                       int32_t *trial_plies, double *vr_mean, double *vr_std_err, double *trial_luck)
{
    // chunks of whole positions; the per-trial results of a chunk go to the caller's arrays or to engine work buffers
    const long long chunk = e->rollout_chunk > 0 ? e->rollout_chunk : kRolloutChunk;
    const long long per_launch = std::max<long long>(1, chunk / trials);
    const long long items_cap = std::min<long long>(n, per_launch) * trials;
    const bool vr = vr_plies >= 0;
    float *sv = nullptr;
    int8_t *so = nullptr;
    int32_t *sp = nullptr;
    double *sl = nullptr;
    int rc;
    if (!trial_value && (rc = e->work.grow(kRolloutValue, (size_t)items_cap * 4, &sv))) return rc;
    if (!trial_outcome && (rc = e->work.grow(kRolloutOutcome, (size_t)items_cap, &so))) return rc;
    if (!trial_plies && (rc = e->work.grow(kRolloutPlies, (size_t)items_cap * 4, &sp))) return rc;
    if (vr && !trial_luck && (rc = e->work.grow(kRolloutLuck, (size_t)items_cap * 8, &sl))) return rc;
    float *rolls = nullptr;
    int4 *zlist = nullptr;
    if (vr && (rc = e->work.grow(kRolloutRolls, (size_t)game_grid(e) * 32 * 32 * 4, &rolls))) return rc;
    if (vr && (rc = e->work.grow(kRolloutZlist, (size_t)game_grid(e) * 32 * 32 * sizeof(int4), &zlist))) return rc;
    RolloutParams p;
    p.trials = trials;
    p.cap = max_plies > 0 ? max_plies : BGX_ROLLOUT_MAX_PLIES;
    p.stratify = (flags & BGX_ROLLOUT_STRATIFY) ? 1 : 0;
    p.seed_lo = (uint32_t)seed; p.seed_hi = (uint32_t)(seed >> 32);
    p.counter = e->counter; p.zstash = e->zstash;
    RolloutVR r = {vr_plies, nullptr, rolls, zlist};
    tick(e);
    for (long long q0 = 0; q0 < n; q0 += per_launch) {
        const long long np = std::min<long long>(n - q0, per_launch);
        const size_t at = (size_t)q0 * trials;
        p.positions = positions + q0 * 32;
        p.n_items = np * trials;
        p.value = trial_value ? trial_value + at : sv;
        p.outcome = trial_outcome ? trial_outcome + at : so;
        p.plies = trial_plies ? trial_plies + at : sp;
        r.luck = trial_luck ? trial_luck + at : sl;
        CU(cudaMemsetAsync(e->counter, 0, sizeof(unsigned long long), e->stream));
        PlyConfigs::dispatch(e->rollout_warps, [&](auto c) {
            constexpr int W = decltype(c)::kWarps, S = decltype(c)::kSets;
            if (vr) k_rollout_vr<W, S><<<game_grid(e), W * 32, ply_smem<W, S>(), e->stream>>>(p, r, e->fixed, e->steal);
            else k_rollout<W, S><<<game_grid(e), W * 32, ply_smem<W, S>(), e->stream>>>(p, e->fixed, e->steal);
        });
        const unsigned grid = (unsigned)((np + 127) / 128);
        if (mean || std_err || counts)
            k_rollout_reduce<<<grid, 128, 0, e->stream>>>(p.value, p.outcome, p.plies, np, trials, mean ? mean + q0 : nullptr,
                                                          std_err ? std_err + q0 : nullptr, counts ? (long long *)counts + q0 * 8 : nullptr);
        e->launches += 2;
        if (vr_mean || vr_std_err) {
            k_rollout_vr_reduce<<<grid, 128, 0, e->stream>>>(p.value, r.luck, np, trials, vr_mean ? vr_mean + q0 : nullptr,
                                                             vr_std_err ? vr_std_err + q0 : nullptr);
            e->launches++;
        }
        CU(cudaGetLastError());
    }
    tock(e);
    return BGX_OK;
}

int bgx_rollout(bgx_engine *e, const int8_t *positions, int64_t n, int32_t trials, int32_t max_plies, uint64_t seed, int flags,
                double *mean, double *std_err, int64_t *counts, float *trial_value, int8_t *trial_outcome, int32_t *trial_plies)
{
    USE(e);
    if (int rc = rollout_args(n, trials, max_plies, flags, "bgx_rollout")) return rc;
    NEED(positions || n == 0, "null positions");
    if (int rc = need_weights(e, "bgx_rollout")) return rc;
    if (n == 0) return BGX_OK;
    return rollout_run(e, positions, n, trials, max_plies, seed, flags, -1, mean, std_err, counts, trial_value, trial_outcome, trial_plies,
                       nullptr, nullptr, nullptr);
}

int bgx_rollout_host(bgx_engine *e, const int8_t *positions, int64_t n, int32_t trials, int32_t max_plies, uint64_t seed, int flags,
                     double *mean, double *std_err, int64_t *counts, float *trial_value, int8_t *trial_outcome, int32_t *trial_plies)
{
    USE(e);
    if (int rc = rollout_args(n, trials, max_plies, flags, "bgx_rollout_host")) return rc;
    NEED(positions || n == 0, "null positions");
    if (int rc = need_weights(e, "bgx_rollout_host")) return rc;
    if (n == 0) return BGX_OK;
    const size_t items = (size_t)n * trials;
    Stage s(e);
    const int8_t *dq = s.in(positions, (size_t)n * 32);
    double *dm = s.out(mean, (size_t)n * 8);
    double *ds = s.out(std_err, (size_t)n * 8);
    int64_t *dc = s.out(counts, (size_t)n * 64);
    float *dv = s.out(trial_value, items * 4);
    int8_t *dout = s.out(trial_outcome, items);
    int32_t *dp = s.out(trial_plies, items * 4);
    if (s.rc) return s.rc;
    return s.finish(bgx_rollout(e, dq, n, trials, max_plies, seed, flags, dm, ds, dc, dv, dout, dp));
}

// ------------------------------------------------------------------------ variance-reduced rollouts (DESIGN 7e)

static int rollout_vr_args(int64_t n, int32_t trials, int32_t max_plies, int flags, int32_t vr_plies, const char *who)
{
    if (int rc = rollout_args(n, trials, max_plies, flags, who)) return rc;
    if (vr_plies < 0 || vr_plies > BGX_ROLLOUT_MAX_PLIES) { set_error("%s: vr_plies must be 0 .. %d", who, BGX_ROLLOUT_MAX_PLIES); return BGX_E_INVALID; }
    return BGX_OK;
}

int bgx_rollout_vr(bgx_engine *e, const int8_t *positions, int64_t n, int32_t trials, int32_t max_plies, uint64_t seed, int flags,
                   int32_t vr_plies, double *mean, double *std_err, int64_t *counts, float *trial_value, int8_t *trial_outcome,
                   int32_t *trial_plies, double *vr_mean, double *vr_std_err, double *trial_luck)
{
    USE(e);
    if (int rc = rollout_vr_args(n, trials, max_plies, flags, vr_plies, "bgx_rollout_vr")) return rc;
    NEED(positions || n == 0, "null positions");
    if (int rc = need_weights(e, "bgx_rollout_vr")) return rc;
    if (n == 0) return BGX_OK;
    return rollout_run(e, positions, n, trials, max_plies, seed, flags, vr_plies, mean, std_err, counts, trial_value, trial_outcome,
                       trial_plies, vr_mean, vr_std_err, trial_luck);
}

int bgx_rollout_vr_host(bgx_engine *e, const int8_t *positions, int64_t n, int32_t trials, int32_t max_plies, uint64_t seed, int flags,
                        int32_t vr_plies, double *mean, double *std_err, int64_t *counts, float *trial_value, int8_t *trial_outcome,
                        int32_t *trial_plies, double *vr_mean, double *vr_std_err, double *trial_luck)
{
    USE(e);
    if (int rc = rollout_vr_args(n, trials, max_plies, flags, vr_plies, "bgx_rollout_vr_host")) return rc;
    NEED(positions || n == 0, "null positions");
    if (int rc = need_weights(e, "bgx_rollout_vr_host")) return rc;
    if (n == 0) return BGX_OK;
    const size_t items = (size_t)n * trials;
    Stage s(e);
    const int8_t *dq = s.in(positions, (size_t)n * 32);
    double *dm = s.out(mean, (size_t)n * 8);
    double *ds = s.out(std_err, (size_t)n * 8);
    int64_t *dc = s.out(counts, (size_t)n * 64);
    float *dv = s.out(trial_value, items * 4);
    int8_t *dout = s.out(trial_outcome, items);
    int32_t *dp = s.out(trial_plies, items * 4);
    double *dvm = s.out(vr_mean, (size_t)n * 8);
    double *dvs = s.out(vr_std_err, (size_t)n * 8);
    double *dl = s.out(trial_luck, items * 8);
    if (s.rc) return s.rc;
    return s.finish(bgx_rollout_vr(e, dq, n, trials, max_plies, seed, flags, vr_plies, dm, ds, dc, dv, dout, dp, dvm, dvs, dl));
}

// the start of a call on lane `lane`: the lane is free, its stream and buffers exist, and its stream waits for the work
// queued on the engine's stream so far (weights set before the call are visible to the lane)
static int lane_begin(bgx_engine *e, int lane, const char *who, bgx_lane **out)
{
    if (lane < 0 || lane >= kLanes) { set_error("%s: lane out of range", who); return BGX_E_INVALID; }
    if (int rc = need_weights(e, who)) return rc;
    bgx_lane &l = e->lanes[lane];
    if (l.busy) { set_error("%s: lane %d has a batch in flight (bgx_lane_wait first)", who, lane); return BGX_E_STATE; }
    if (!l.stream) {
        CU(cudaStreamCreateWithFlags(&l.stream, cudaStreamNonBlocking));
        CU(cudaEventCreateWithFlags(&l.done, cudaEventDisableTiming));
        CU(cudaMalloc(&l.counter, kCounterBytes));
        CU(cudaMalloc(&l.steal, (size_t)e->sm_count * 32 * kStealMaxResults * sizeof(StealResult)));
    }
    CU(cudaEventRecord(e->ev_sync, e->stream));
    CU(cudaStreamWaitEvent(l.stream, e->ev_sync, 0));
    *out = &l;
    return BGX_OK;
}

// Asynchronous form of bgx_select_moves_host: the copies and the kernel are queued on lane `lane`'s own
// stream and the call returns; bgx_lane_wait blocks until that lane's results are in the host buffers.
// A few lanes in flight let the host advance one part of a population while the GPU plays the others.
int bgx_select_moves_host_async(bgx_engine *e, int lane, const int8_t *queries, int64_t n, float epsilon, uint64_t seed,
                                int8_t *chosen, int8_t *moves, int8_t *moves_len, float *value, int32_t *n_seq, int32_t *n_scored)
{
    USE(e);
    NEED(queries && n >= 0, "bad argument");
    bgx_lane *l;
    if (int rc = lane_begin(e, lane, "bgx_select_moves_host_async", &l)) return rc;
    if (n == 0) return BGX_OK;
    OrderPlan plan;
    if (n <= e->select_order_max) {
        if (int rc = l->work.grow(kLaneOrder0, (size_t)n * kOrderBuckets * 4, &plan.region[0])) return rc;
    }
    l->order_n = -1;
    Stage s(*l);
    const int8_t *dq = s.in(queries, (size_t)n * 32);
    const SelectOut out = {s.out(chosen, (size_t)n * 32), s.out(moves, (size_t)n * 8), s.out(moves_len, (size_t)n),
                           s.out(value, (size_t)n * 4), s.out(n_seq, (size_t)n * 4), s.out(n_scored, (size_t)n * 4)};
    if (s.rc) return s.rc;
    return s.finish(launch_select(e, l->stream, l->counter, l->steal, dq, n, epsilon, seed, out, plan, e->lane_grid));
}

static int play_ply(bgx_engine *e, int lane, const int8_t *records, int32_t *ply, int64_t *game_id, int64_t id_stride, int first_mover,
                    int64_t n, float epsilon, uint64_t explore_seed, uint64_t dice_seed,
                    int8_t *next_records, int8_t *winner, float *value, int32_t *n_seq, const char *who)
{
    NEED(records && next_records && n >= 0, "bad argument");
    bgx_lane *l;
    if (int rc = lane_begin(e, lane, who, &l)) return rc;
    if (n == 0) return BGX_OK;
    OrderPlan plan;
    if (n <= e->select_order_max) {
        const void *before[2] = {l->work.buf[kLaneOrder0], l->work.buf[kLaneOrder1]};
        int rc;
        if ((rc = l->work.grow(kLaneOrder0, (size_t)n * kOrderBuckets * 4, &plan.region[0]))) return rc;
        if ((rc = l->work.grow(kLaneOrder1, (size_t)n * kOrderBuckets * 4, &plan.region[1]))) return rc;
        if (before[0] != plan.region[0] || before[1] != plan.region[1]) l->order_n = -1;   // reallocated: the stored queue is gone
        plan.slot = l->order_slot;
        plan.ready = l->order_n == n;          // the previous call on this lane sorted ITS outputs for us: if the caller's
        plan.produce = true;                   // queries are something else the order is merely a poor one, never wrong
    }
    Stage s(*l);
    const int8_t *dq = s.in(records, (size_t)n * 32);
    int32_t *dp = s.in(ply, (size_t)n * 4);
    long long *dg = s.in((long long *)game_id, (size_t)n * 8);
    int8_t *dc = s.out(next_records, (size_t)n * 32);
    int8_t *dw = s.out(winner, (size_t)n);
    const SelectOut out = {nullptr, nullptr, nullptr, s.out(value, (size_t)n * 4), s.out(n_seq, (size_t)n * 4), nullptr};
    if (id_stride > 0) {                       // restart mode: the kernel updates ply and game id in place
        s.copy_back(ply, dp, (size_t)n * 4);
        s.copy_back(game_id, dg, (size_t)n * 8);
    }
    if (s.rc) return s.rc;
    AdvanceOut adv = {dc, dw, dp, dg, (uint32_t)dice_seed, (uint32_t)(dice_seed >> 32), nullptr, nullptr,
                      (long long)id_stride, first_mover, id_stride > 0 ? dp : nullptr, id_stride > 0 ? dg : nullptr};
    if (int rc = launch_select(e, l->stream, l->counter, l->steal, dq, n, epsilon, explore_seed, out, plan, e->lane_grid, adv)) return rc;
    if (plan.produce) { l->order_slot = 1 - plan.slot; l->order_n = n; }
    return s.finish();
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
    if (int rc = need_weights(e, "self-play")) return rc;
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
    PlyConfigs::dispatch(e->selfplay_warps, [&](auto c) {
        constexpr int W = decltype(c)::kWarps, S = decltype(c)::kSets;
        dispatch_explore(epsilon > 0.f, [&](auto x) {
            k_selfplay<W, S, decltype(x)::value><<<game_grid(e), W * 32, ply_smem<W, S>(), e->stream>>>(p, e->fixed, e->flat, e->steal);
        });
    });
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
    Stage s(e);
    int8_t *d = s.out(records, (size_t)e->n_slots * per_game * 32);
    if (s.rc) return s.rc;
    return s.finish(bgx_selfplay_sample(e, per_game, seed, d));
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
    if (int rc = need_weights(e, "TD replay")) return rc;
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
    if (int rc = need_weights(e, "bgx_td_replay_host")) return rc;
    int8_t slot[32] = {0};
    slot[31] = player1_won ? kP1Won : kP2Won;
    std::vector<float> flat(BGX_NPARAMS_PADDED);
    Stage s(e);
    const int8_t *dtraj = s.in(records, (size_t)T * 32);
    const int8_t *dslot = s.in(slot, 32);
    const int32_t *dply = s.in(&T, 4);
    float *dfinal = s.out(flat.data(), flat.size() * sizeof(float));
    double *dsq = s.take<double>((size_t)T * 8);
    if (s.rc) return s.rc;
    if (sq_errors && T > 1) s.copy_back(sq_errors, dsq, (size_t)(T - 1) * 8);
    CU(cudaMemsetAsync(dsq, 0, (size_t)T * 8, e->stream));
    if (int rc = s.finish(launch_td(e, dtraj, dslot, dply, 1, T, lr, lambda, -1, nullptr, dfinal, dsq, nullptr))) return rc;
    unpack_weights(flat.data(), new_W1, new_b1, new_w2, new_b2);
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
