// bgx_kernels.cuh — the __global__ kernels of libbgx (sm_100a).  See bgx_device.cuh for
// the execution model; DESIGN.md for the roofline of each kernel.
#pragma once
#include "bgx_device.cuh"
#include "bgx_ply.cuh"

namespace bgx {

constexpr int kGameWarps = 16;                     // warps per CTA in the warp-per-position kernels
constexpr int kGameThreads = kGameWarps * 32;
// what a self-play warp knows about the slot it is seated at, apart from the position itself: kept in shared
// memory (lane 0 writes, __syncwarp, everybody reads) to leave the registers to the walk
struct WarpSeat {
    long long slot;
    unsigned long long gid;
    int ply, step, status, player;
    int carry;                                     // the warp's stash holds the pre-activation of the slot's position (greedy_ply)
    int dice_base;                                 // lane l holds the dice of ply dice_base + l of the slot's game (-1: nothing held)
};

// dynamic shared memory of the fused ply kernels: weight table + per-warp scratch + sharing slots + seats + barrier
template <int kWarps, int kSets>
constexpr int ply_smem()
{
    return kFixedBytes + kWarps * (int)sizeof(PlyScratch<kSets>) + (int)sizeof(StealShared<kWarps>) + kWarps * (int)sizeof(WarpSeat) + 16;
}

// the launch configurations of the fused ply kernels (k_select, k_selfplay, k_rollout): warps per CTA and the cache sets per
// warp that fill the shared memory at that width.  Each kernel is instantiated once per entry.
template <int W, int S>
struct PlyConfig {
    static constexpr int kWarps = W, kSets = S, kSmem = ply_smem<W, S>();
};
template <typename... C>
struct PlyConfigList {
    static constexpr bool has(long long warps) { return ((warps == C::kWarps) || ...); }
    static constexpr bool fits(int smem_bytes) { return ((C::kSmem <= smem_bytes) && ...); }
    // f(config) for every configuration, stopping at the first non-zero result, which is returned
    template <typename F>
    static int each(F &&f)
    {
        int rc = 0;
        ((rc = rc ? rc : f(C{})), ...);
        return rc;
    }
    // f(config) for the configuration with `warps` warps per CTA
    template <typename F>
    static void dispatch(int warps, F &&f) { ((warps == C::kWarps ? f(C{}) : void()), ...); }
};
using PlyConfigs = PlyConfigList<PlyConfig<16, 109>, PlyConfig<20, 86>, PlyConfig<24, 72>, PlyConfig<32, 53>>;
constexpr int kEvalSmem = kFixedBytes + 16;            // k_evaluate: table + barrier

// exact-dedup table of the summary kernel: per warp, in global memory (L2 resident)
constexpr int kUniqSlots = 4096;                   // 8 words each, probed as buckets of 4 slots
constexpr int kUniqWords = 8;
constexpr size_t kUniqBytesPerWarp = (size_t)kUniqSlots * kUniqWords * 4;   // 128 KiB

// ---- weights: state_dict order -> the tables the kernels read ------------------------------
// flat = [W1[128][198] | b1[128] | w2[128] | b2[1]]  (model.py:36-37)
// Wt[198][128]: W1 transposed (feature-major), fp32, for the TD kernel
__global__ void k_build_table(const float *__restrict__ flat, float *__restrict__ Wt)
{
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= kTableFloats) return;
    const int f = idx / kHidden, j = idx % kHidden;
    Wt[idx] = flat[j * kFeatures + f];
}

// aux[0] = S, aux[1] = 1/S: the fixed-point scale of the ply evaluator (bgx_ply.cuh).  Thread j bounds
// |z_j| over every position: |b1_j| + per point the largest contribution any stack of either colour can make
// (up to 15 checkers: three unit features and a slope of up to 6) + both bars at 7.5 + both borne-off
// features at 1 + the larger turn flag.  S = the largest power of two with max_j bound_j * S <= 2^30.
__global__ void k_fixed_scale(const float *__restrict__ flat, float *__restrict__ aux)
{
    __shared__ float red[kHidden / 32];
    const int j = threadIdx.x;
    const float *w = flat + j * kFeatures;
    float bound = fabsf(flat[kTableFloats + j]);
    for (int i = 0; i < 24; i++) {
        float worst = 0.f;
        for (int c = 0; c < 2; c++) {
            const float *u = w + 8 * i + 4 * c;
            const float s1 = u[0], s2 = s1 + u[1], s3 = s2 + u[2];
            worst = fmaxf(worst, fmaxf(fabsf(s1), fabsf(s2)));
            worst = fmaxf(worst, fabsf(s3) + 6.f * fabsf(u[3]));
        }
        bound += worst;
    }
    bound += fmaxf(fabsf(w[192]), fabsf(w[193])) + 7.5f * (fabsf(w[194]) + fabsf(w[195])) + fabsf(w[196]) + fabsf(w[197]);
    // the output sum y = w2 . h (|y| <= sum |w2_j|, h in (0, 1)) is reduced over the warp as an INTEGER too (one REDUX.SUM,
    // order-independent like z): scale Y = the largest power of two with sum_j |w2_j| * Y <= 2^30
    float w2sum = fabsf(flat[kTableFloats + kHidden + j]);
    for (int o = 16; o > 0; o >>= 1) {
        bound = fmaxf(bound, __shfl_xor_sync(kFull, bound, o));
        w2sum += __shfl_xor_sync(kFull, w2sum, o);
    }
    __shared__ float red2[kHidden / 32];
    if ((j & 31) == 0) { red[j >> 5] = bound; red2[j >> 5] = w2sum; }
    __syncthreads();
    if (j == 0) {
        for (int k = 1; k < kHidden / 32; k++) { bound = fmaxf(bound, red[k]); w2sum += red2[k]; }
        int e = 30 - (ilogbf(fmaxf(bound, 1e-30f)) + 1);      // bound < 2^(ilogb+1)  =>  bound * 2^e < 2^30
        e = e > 60 ? 60 : (e < -60 ? -60 : e);
        aux[0] = ldexpf(1.f, e);
        aux[1] = ldexpf(1.f, -e);
        aux[2] = bound;
        int ey = 30 - (ilogbf(fmaxf(w2sum, 1e-30f)) + 1);
        ey = ey > 40 ? 40 : (ey < -60 ? -60 : ey);
        aux[3] = ldexpf(1.f, ey);
    }
}

// Ti[228][128]: the fixed-point table of the ply evaluator (layout in bgx_ply.cuh)
__global__ void k_build_fixed(const float *__restrict__ flat, const float *__restrict__ aux, int32_t *__restrict__ Ti)
{
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= kFixedInts) return;
    const int f = idx / kHidden, j = idx % kHidden;
    const float S = aux[0];
    if (f < kFeatures) {
        const float w = flat[j * kFeatures + f];
        const bool half = (f < 192 && (f & 3) == 3) || f == 194 || f == 195;
        Ti[idx] = f >= 196 ? __float_as_int(w) : __float2int_rn(w * (half ? 0.5f * S : S));
    } else if (f < kRowB1) {                       // row 198 + 15 p + k: what the (k+1)-th borne-off checker of player p adds
        const int p = (f - kFeatures) / 15, k = (f - kFeatures) % 15;
        const float w = flat[j * kFeatures + 196 + p];
        Ti[idx] = __float2int_rn(w * (kOffFeature[k + 1] * S)) - __float2int_rn(w * (kOffFeature[k] * S));
    } else if (f == kRowB1) {
        Ti[idx] = __float2int_rn(flat[kTableFloats + j] * S);
    } else if (f == kRowW2) {
        Ti[idx] = __float_as_int(flat[kTableFloats + kHidden + j]);
    } else if (f == kRowConst) {                   // constants, the same float4 for every lane
        const float c[4] = {S, -1.4426950408889634f * aux[1], flat[kTableFloats + 2 * kHidden], aux[3]};
        Ti[idx] = __float_as_int(c[j & 3]);
    } else {                                       // what depends on the lane only: read where needed instead of held (or recomputed) in registers
        Ti[idx] = j < 32 ? (int32_t)ply_hash_multiplier(j) : 0;       // word l of the row: lane l's multiplier (one bank per lane)
    }
}

// a warp-wide work queue: lane 0 claims, everybody learns
__device__ __forceinline__ long long claim(unsigned long long *counter, int lane)
{
    unsigned long long i = 0;
    if (lane == 0) i = atomicAdd(counter, 1ull);
    return (long long)__shfl_sync(kFull, i, 0);
}

// one 32-byte record per warp: lane i gets byte i
__device__ __forceinline__ int load_record_byte(const int8_t *rec, int lane) { return (int)rec[lane]; }

// ---- batched evaluateTurnSequences, summary form (cppsrc/game.cpp:193-222) -------------
struct SummaryLeaf {
    uint32_t *table;       // this warp's exact-dedup table (global)
    uint32_t gen;
    int lane;
    int n_seq = 0, n_unique = 0;
    bool overflow = false;
    uint64_t digest = 0;

    __device__ __forceinline__ void operator()(int v, uint64_t moves, int)
    {
        uint32_t k[5];
        key_planes(v, k);
        n_seq++;
        digest = digest * kDigestMul + leaf_hash(k, moves);
        if (overflow) return;
        // bucket of 4 slots x 8 words = one 128-byte line; lane l looks at word l%8 of slot l/8
        const uint32_t k4g = k[4] | (gen << 24);
        const int w = lane & 7;
        const uint32_t mine = w == 0 ? k[0] : w == 1 ? k[1] : w == 2 ? k[2] : w == 3 ? k[3] : k4g;
        uint32_t bucket = hash_planes(k) & (kUniqSlots / 4 - 1);
        for (int probe = 0; probe < kUniqSlots / 4; probe++) {
            uint32_t *line = table + (size_t)bucket * 32;
            const uint32_t got = line[lane];
            const uint32_t same = __ballot_sync(kFull, w >= 5 || got == mine);
            const uint32_t stale = __ballot_sync(kFull, w == 4 && (got >> 24) != gen);
            for (int s = 0; s < 4; s++) {
                if (((same >> (8 * s)) & 0xFFu) == 0xFFu) return;              // seen before
                if ((stale >> (8 * s + 4)) & 1u) {                              // first free slot: insert
                    if ((lane >> 3) == s && w < 5) line[lane] = mine;
                    __syncwarp();
                    n_unique++;
                    return;
                }
            }
            bucket = (bucket + 1) & (kUniqSlots / 4 - 1);
        }
        overflow = true;
    }
};

__global__ void __launch_bounds__(kGameThreads, 1)
k_enumerate_summary(const int8_t *__restrict__ queries, long long n, int32_t *__restrict__ n_seq,
                    int32_t *__restrict__ n_unique, unsigned long long *__restrict__ digest,
                    uint32_t *__restrict__ tables, uint32_t *__restrict__ gens, unsigned long long *counter)
{
    const int lane = threadIdx.x & 31;
    const int gwarp = blockIdx.x * (blockDim.x >> 5) + warp_index();
    uint32_t *table = tables + (size_t)gwarp * (kUniqBytesPerWarp / 4);
    uint32_t gen = gens[gwarp];                     // the table outlives the launch, so does its generation
    for (;;) {
        const long long q = claim(counter, lane);
        if (q >= n) break;
        const int b = load_record_byte(queries + q * 32, lane);
        const int root = lane < 28 ? b : 0;
        const int player = __shfl_sync(kFull, b, 28), d1 = __shfl_sync(kFull, b, 29), d2 = __shfl_sync(kFull, b, 30);
        gen = (gen + 1) & 0xFFu;
        if (gen == 0) {
            for (int i = lane; i < kUniqSlots * kUniqWords; i += 32) table[i] = 0;
            gen = 1;
            __syncwarp();
        }
        SummaryLeaf leaf;
        leaf.table = table; leaf.gen = gen; leaf.lane = lane;
        walk_turn(root, lane, player, d1, d2, leaf);
        if (lane == 0) {
            n_seq[q] = leaf.n_seq;
            n_unique[q] = leaf.overflow ? -1 : leaf.n_unique;
            digest[q] = leaf.digest;
        }
        __syncwarp();                               // reconverged before the back-edge (see k_selfplay)
    }
    if (lane == 0) gens[gwarp] = gen;
}

// ---- batched legalTurnSequences, count only (game.cpp:134-191): the size of every query's list ----
__global__ void __launch_bounds__(kGameThreads, 1)
k_enumerate_count(const int8_t *__restrict__ queries, long long n, int32_t *__restrict__ n_seq, unsigned long long *counter)
{
    const int lane = threadIdx.x & 31;
    for (;;) {
        const long long q = claim(counter, lane);
        if (q >= n) break;
        const int b = load_record_byte(queries + q * 32, lane);
        const int root = lane < 28 ? b : 0;
        const int player = __shfl_sync(kFull, b, 28), d1 = __shfl_sync(kFull, b, 29), d2 = __shfl_sync(kFull, b, 30);
        CountLeaf leaf;
        walk_turn(root, lane, player, d1, d2, leaf);
        if (lane == 0) n_seq[q] = leaf.n;
        __syncwarp();                               // reconverged before the back-edge (see k_selfplay)
    }
}

// ---- exclusive prefix sum of the counts (int32 -> int64 offsets[n + 1]) in three small launches ----
constexpr int kScanThreads = 256, kScanPerThread = 8, kScanTile = kScanThreads * kScanPerThread;

__device__ __forceinline__ long long block_exclusive_scan(long long x, long long *warp_sums, long long &block_total)
{
    const int lane = threadIdx.x & 31, warp = warp_index(), n_warps = blockDim.x >> 5;
    long long inc = x;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const long long y = __shfl_up_sync(kFull, inc, o);
        if (lane >= o) inc += y;
    }
    if (lane == 31) warp_sums[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        const long long s = lane < n_warps ? warp_sums[lane] : 0;
        long long si = s;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long y = __shfl_up_sync(kFull, si, o);
            if (lane >= o) si += y;
        }
        if (lane < n_warps) warp_sums[lane] = si - s;
        if (lane == 31) warp_sums[32] = si;
    }
    __syncthreads();
    block_total = warp_sums[32];
    const long long base = warp_sums[warp];
    __syncthreads();
    return base + inc - x;
}

__global__ void __launch_bounds__(kScanThreads) k_scan_tiles(const int32_t *__restrict__ cnt, long long n, long long *__restrict__ offsets,
                                                           long long *__restrict__ tile_sums)
{
    __shared__ long long warp_sums[33];
    const long long first = (long long)blockIdx.x * kScanTile + (long long)threadIdx.x * kScanPerThread;
    long long v[kScanPerThread], mine = 0;
#pragma unroll
    for (int i = 0; i < kScanPerThread; i++) {
        v[i] = first + i < n ? (long long)cnt[first + i] : 0;
        mine += v[i];
    }
    long long total;
    long long run = block_exclusive_scan(mine, warp_sums, total);
#pragma unroll
    for (int i = 0; i < kScanPerThread; i++) {
        if (first + i < n) offsets[first + i] = run;
        run += v[i];
    }
    if (threadIdx.x == 0) tile_sums[blockIdx.x] = total;
}

__global__ void __launch_bounds__(1024) k_scan_sums(long long *__restrict__ tile_sums, int n_tiles)
{
    __shared__ long long warp_sums[33];
    long long carry = 0;
    for (int base = 0; base < n_tiles; base += 1024) {
        const int i = base + threadIdx.x;
        const long long x = i < n_tiles ? tile_sums[i] : 0;
        long long total;
        const long long ex = block_exclusive_scan(x, warp_sums, total);
        if (i < n_tiles) tile_sums[i] = carry + ex;
        carry += total;
    }
    if (threadIdx.x == 0) tile_sums[n_tiles] = carry;
}

__global__ void __launch_bounds__(kScanThreads) k_scan_add(long long *__restrict__ offsets, long long n, const long long *__restrict__ tile_sums, int n_tiles)
{
    const long long i = (long long)blockIdx.x * kScanThreads + threadIdx.x;
    if (i < n) offsets[i] += tile_sums[i / kScanTile];
    if (i == 0) offsets[n] = tile_sums[n_tiles];
}

// ---- batched evaluateTurnSequences, materialised (game.cpp:193-222, bindings:27-39) ----
struct WriteLeaf {
    int8_t *moves, *lens, *states;   // already offset to this query's first row
    int lane, player;
    long long row = 0;
    __device__ __forceinline__ void operator()(int v, uint64_t mv, int len)
    {
        int8_t *st = states + row * 32;
        const int out = lane < 28 ? v : (lane == 28 ? player : 0);
        st[lane] = (int8_t)out;                                        // one 32-byte sector per sequence
        if (lane < 8) {
            const int j = lane >> 1;
            const int code = (int)((mv >> (10 * j + 5 * (lane & 1))) & 31u);
            moves[row * 8 + lane] = (int8_t)(j < len ? code : 0);
        }
        if (lane == 8) lens[row] = (int8_t)len;
        row++;
        __syncwarp();                                                  // the walk's loop continues from here: reconverged (see k_selfplay)
    }
};

__global__ void __launch_bounds__(kGameThreads, 1)
k_enumerate_write(const int8_t *__restrict__ queries, long long n, const long long *__restrict__ offsets,
                  int8_t *__restrict__ seq_moves, int8_t *__restrict__ seq_len, int8_t *__restrict__ states,
                  unsigned long long *counter)
{
    const int lane = threadIdx.x & 31;
    for (;;) {
        const long long q = claim(counter, lane);
        if (q >= n) break;
        const int b = load_record_byte(queries + q * 32, lane);
        const int root = lane < 28 ? b : 0;
        const int player = __shfl_sync(kFull, b, 28), d1 = __shfl_sync(kFull, b, 29), d2 = __shfl_sync(kFull, b, 30);
        const long long base = offsets[q];
        WriteLeaf leaf;
        leaf.moves = seq_moves + base * 8; leaf.lens = seq_len + base; leaf.states = states + base * 32;
        leaf.lane = lane; leaf.player = player;
        walk_turn(root, lane, player, d1, d2, leaf);
    }
}

// ---- _encode_states_np (model.py:111-144): records -> fp32 [n][198], HBM-bound -----------
// A CTA builds a tile of kEncRows rows (kEncRows * 792 B, contiguous in X and a 16-byte multiple starting
// on a 16-byte boundary because tiles start on even rows) in shared memory and hands it to the TMA engine:
// one cp.async.bulk.global.shared per tile (SASS UBLKCP), two tiles in flight per CTA, so the store
// stream costs the SM one instruction per 25 KB and overlaps the encoding of the next tile.
constexpr int kEncWarps = 8;
constexpr int kEncRows = 32;                        // rows per tile (4 per warp)
constexpr int kEncTileFloats = kEncRows * kFeatures;
constexpr int kEncSmem = 2 * kEncTileFloats * 4;    // 50,688 B

__global__ void __launch_bounds__(kEncWarps * 32)
k_encode(const int8_t *__restrict__ records, long long n, float *__restrict__ X)
{
    extern __shared__ __align__(128) float enc_tiles[];
    const int lane = threadIdx.x & 31, warp = warp_index();
    const long long n_tiles = (n + kEncRows - 1) / kEncRows;
    int buf = 0;
    for (long long t = blockIdx.x; t < n_tiles; t += gridDim.x, buf ^= 1) {
        float *tile = enc_tiles + buf * kEncTileFloats;
        // the bulk store that last read this buffer (two tiles ago) must have finished reading it
        if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
        __syncthreads();
        const long long row0 = t * kEncRows;
        // 4 records (128 B) per warp in one coalesced 4-byte-per-lane load
        const long long r_first = row0 + warp * 4;
        int word = 0;
        {
            const long long byte = r_first * 32 + lane * 4;
            if (byte + 3 < n * 32) word = *reinterpret_cast<const int *>(records + byte);
        }
#pragma unroll
        for (int r = 0; r < 4; r++) {
            const int w = __shfl_sync(kFull, word, r * 8 + (lane >> 2));
            const int v = (int)(int8_t)(w >> (8 * (lane & 3)));        // byte `lane` of record r
            // every lane encodes the element it holds: lanes 0..23 a point (8 features), 24..27 a bar / borne-off
            // count (1 feature), 28 the turn flag (2 features); no cross-lane traffic, no divergent slow paths
            float *row = tile + (warp * 4 + r) * kFeatures;
            if (lane < 24) {
                const int c = v < 0 ? -v : v;
                const float a = c >= 1 ? 1.f : 0.f, b = c >= 2 ? 1.f : 0.f, cc = c >= 3 ? 1.f : 0.f;
                const float d = c >= 4 ? (float)(c - 3) * 0.5f : 0.f;
                float2 *dst = reinterpret_cast<float2 *>(row + 8 * lane);   // 8-byte aligned always
                const bool p1 = v > 0;
                dst[0] = p1 ? make_float2(a, b) : make_float2(0.f, 0.f);
                dst[1] = p1 ? make_float2(cc, d) : make_float2(0.f, 0.f);
                dst[2] = p1 ? make_float2(0.f, 0.f) : make_float2(a, b);
                dst[3] = p1 ? make_float2(0.f, 0.f) : make_float2(cc, d);
            } else if (lane < 28) {
                row[170 + lane] = lane < 26 ? (float)v * 0.5f : kOffFeature[v & 15];
            } else if (lane == 28) {
                *reinterpret_cast<float2 *>(row + 192) = v == 0 ? make_float2(1.f, 0.f) : make_float2(0.f, 1.f);
            }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // generic-proxy writes -> visible to the TMA engine
        __syncthreads();
        const long long rows_here = (n - row0) < kEncRows ? (n - row0) : kEncRows;
        float *out = X + row0 * kFeatures;
        const int bulk_rows = (int)rows_here & ~1;                        // an even number of rows is a 16-byte multiple
        if (threadIdx.x == 0) {
            if (bulk_rows > 0)
                asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                             ::"l"(out), "r"(smem_u32(tile)), "r"(bulk_rows * kFeatures * 4)
                             : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
        if (rows_here & 1) {                                              // the odd last row of the whole array
            const int base = bulk_rows * kFeatures;
            for (int i = threadIdx.x; i < kFeatures; i += blockDim.x) out[base + i] = tile[base + i];
        }
    }
    if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

// ---- forward(_encode_states_np(states, turn)) (model.py:63-67): records -> V ------------
__global__ void __launch_bounds__(kGameThreads, 1)
k_evaluate(const int8_t *__restrict__ records, long long n, float *__restrict__ V,
           const int32_t *__restrict__ Ti, const float *__restrict__ flat)
{
    extern __shared__ __align__(128) unsigned char smem[];
    int32_t *sT = reinterpret_cast<int32_t *>(smem);
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem + kFixedBytes);
    stage_table(sT, Ti, bar, kFixedBytes);
    const int lane = threadIdx.x & 31;
    PlyEvaluator ev;
    ev.T4 = reinterpret_cast<const int4 *>(sT);
    const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
    for (long long q = (long long)blockIdx.x * (blockDim.x >> 5) + warp_index(); q < n; q += warps) {
        const int b = load_record_byte(records + q * 32, lane);
        const int v = lane < 28 ? b : 0;
        const float val = ev.finish(ev.preactivation(v, lane, __shfl_sync(kFull, b, 28) ? 1 : 0), lane);
        if (lane == 0) V[q] = val;
    }
}

// ---- batched make_move (model.py:180-222) ------------------------------------------------
struct SelectOut {
    int8_t *chosen, *moves, *moves_len;
    float *value;
    int32_t *n_seq, *n_scored;
};

__device__ __forceinline__ void store_choice(const SelectOut &o, long long q, const Choice &c, int lane, int player)
{
    const int len = (int)(c.moves >> 40);
    if (o.chosen) {
        const int out = lane < 28 ? c.v : (lane == 28 ? player : (lane == 31 ? (len > 0 ? 1 : 0) : 0));
        o.chosen[q * 32 + lane] = (int8_t)out;
    }
    if (o.moves && lane < 8) {
        const int j = lane >> 1;
        const int code = (int)((c.moves >> (10 * j + 5 * (lane & 1))) & 31u);
        o.moves[q * 8 + lane] = (int8_t)(j < len ? code : 0);
    }
    if (lane == 0) {
        if (o.moves_len) o.moves_len[q] = (int8_t)len;
        if (o.value) o.value[q] = c.value;
        if (o.n_seq) o.n_seq[q] = c.n_seq;
        if (o.n_scored) o.n_scored[q] = c.n_scored;
    }
}

// shared-memory carve-up of the fused ply kernels: weight table | per-warp caches | sharing slots | seats | barrier
template <int kWarps, int kSets>
struct PlySmem {
    int32_t *table;
    PlyScratch<kSets> *scratch;
    StealShared<kWarps> *share;
    WarpSeat *seat;
    uint64_t *bar;
    __device__ __forceinline__ explicit PlySmem(unsigned char *smem)
    {
        table = reinterpret_cast<int32_t *>(smem);
        scratch = reinterpret_cast<PlyScratch<kSets> *>(smem + kFixedBytes);
        share = reinterpret_cast<StealShared<kWarps> *>(smem + kFixedBytes + kWarps * sizeof(PlyScratch<kSets>));
        seat = reinterpret_cast<WarpSeat *>(smem + kFixedBytes + kWarps * sizeof(PlyScratch<kSets>) + sizeof(StealShared<kWarps>));
        bar = reinterpret_cast<uint64_t *>(smem + kFixedBytes + kWarps * sizeof(PlyScratch<kSets>) + sizeof(StealShared<kWarps>) +
                                           kWarps * sizeof(WarpSeat));
    }
    // every thread calls this before stage_table(), whose __syncthreads publishes it
    __device__ __forceinline__ void init_share() const
    {
        if (threadIdx.x < kWarps) {
            share->slot[threadIdx.x].legal0 = 0;
            share->slot[threadIdx.x].pending = 0;
            share->slot[threadIdx.x].nres = 0;
        }
        if (threadIdx.x == 0) share->pad[0] = 0;
        if (threadIdx.x == 0) { share->active = kWarps; share->urgent = 0; }
        if (threadIdx.x < 8) share->stats[threadIdx.x] = 0;
    }
};

// ---- queue order of a one-ply launch ----------------------------------------------------------------------
// A one-ply launch over a few ten thousand queries is as long as its tail: turn trees range from 0 to ~12 k
// sequences.  k_select_order sorts the queue heaviest first by a cheap estimate of the tree size (counting sort
// into 16 power-of-two buckets): root origins k of each die, taken once as they are and - with checkers on the bar -
// once more with the bar emptied (after the entries the turn goes on freely).  The order only decides WHEN a query
// is walked, never its result (values are pure functions of the query).
constexpr int kOrderBuckets = 16;
constexpr int kOrderCtaQueries = 64;     // 8 warps x 8 queries

__device__ __forceinline__ int order_bucket(int v, int lane, int player, int d1, int d2)
{
    const Mover m(lane, player);
    const int bar = __shfl_sync(kFull, v, 24 + player);
    const int k1 = __popc(m.legal_here(v, d1));
    const int k2 = d1 == d2 ? k1 : __popc(m.legal_here(v, d2));
    long long est;
    if (bar == 0) {
        est = d1 == d2 ? (long long)k1 * k1 * k1 * k1 : 2ll * k1 * k2 + k1 + k2;
    } else {
        const int vf = lane == 24 + player ? 0 : v;
        const int f1 = __popc(m.legal_here(vf, d1)) + 1;
        const int f2 = d1 == d2 ? f1 : __popc(m.legal_here(vf, d2)) + 1;
        if (d1 == d2) {
            est = k1;
            for (int j = bar; j < 4; j++) est *= f1;
        } else {
            est = bar == 1 ? (long long)k1 * f2 + (long long)k2 * f1 + k1 + k2 : (long long)k1 * k2;
        }
    }
    const int b = 63 - __clzll(est + 1);
    return b < kOrderBuckets ? b : kOrderBuckets - 1;
}

// region[b][..totals[b]] = the queries of bucket b (any order inside a bucket); totals zeroed by the caller
__global__ void __launch_bounds__(256) k_select_order(const int8_t *__restrict__ queries, long long n, int32_t *__restrict__ region,
                                                      uint32_t *__restrict__ totals)
{
    __shared__ uint32_t hist[kOrderBuckets], base[kOrderBuckets];
    __shared__ uint8_t key[kOrderCtaQueries];
    const int lane = threadIdx.x & 31, warp = warp_index();
    const long long q0 = (long long)blockIdx.x * kOrderCtaQueries;
    if (threadIdx.x < kOrderBuckets) hist[threadIdx.x] = 0;
    __syncthreads();
    for (int j = warp; j < kOrderCtaQueries; j += 8) {
        const long long q = q0 + j;
        if (q >= n) break;
        const int b = load_record_byte(queries + q * 32, lane);
        const int player = __shfl_sync(kFull, b, 28) ? 1 : 0, d1 = __shfl_sync(kFull, b, 29), d2 = __shfl_sync(kFull, b, 30);
        const int k = order_bucket(lane < 28 ? b : 0, lane, player, d1, d2);
        if (lane == 0) { key[j] = (uint8_t)k; atomicAdd(&hist[k], 1u); }
    }
    __syncthreads();
    if (threadIdx.x < kOrderBuckets) {
        const uint32_t c = hist[threadIdx.x];
        base[threadIdx.x] = c ? atomicAdd(&totals[threadIdx.x], c) : 0u;
        hist[threadIdx.x] = 0;
    }
    __syncthreads();
    if (threadIdx.x < kOrderCtaQueries && q0 + threadIdx.x < n) {
        const int k = key[threadIdx.x];
        region[(size_t)k * n + base[k] + atomicAdd(&hist[k], 1u)] = (int32_t)(q0 + threadIdx.x);
    }
}

// bgx_play_ply_host_async: the rest of the ply (k_advance's work) done by the warp that chose the move, and the
// bucket of the NEXT ply's query appended to the sorted queue of the lane's next launch - one kernel per ply-step,
// no small kernels that would wait for an SM behind the persistent ones.
struct AdvanceOut {
    int8_t *next;                 // [n][32] advanced records (nullptr: plain select)
    int8_t *winner;               // [n] or nullptr
    const int32_t *ply_of;        // [n] ply whose dice each game gets (restart mode: the ply just played), or nullptr (0)
    const long long *game_id;     // [n] or nullptr (the query index)
    uint32_t seed_lo, seed_hi;    // dice key
    int32_t *next_region;         // [16][n] or nullptr
    uint32_t *next_totals;        // [16], zeroed by the caller
    // restart mode (id_stride > 0): a finished game is replaced in place by the opening record of game id + id_stride,
    // and the ply / game id of what `next` now holds are written back (the buffers may be ply_of / game_id themselves)
    long long id_stride;
    int first_mover;
    int32_t *ply_out;
    long long *gid_out;
};

__device__ __forceinline__ void store_advanced(const AdvanceOut &a, long long q, long long n, int v, int lane, int player)
{
    const int off1 = __shfl_sync(kFull, v, 26), off2 = __shfl_sync(kFull, v, 27);
    const int win = off1 == 15 ? 0 : (off2 == 15 ? 1 : -1);                  // game.cpp:388-407
    unsigned long long g = a.game_id ? (unsigned long long)a.game_id[q] : (unsigned long long)q;
    int ply = a.ply_of ? a.ply_of[q] : 0;
    int mover = win < 0 ? player ^ 1 : player, status = win + 1;
    if (a.id_stride > 0) {
        ply++;
        if (win >= 0) {                                                      // train.py:64-97 for the slot's next game
            g += (unsigned long long)a.id_stride;
            ply = 0;
            v = start_value(lane);
            mover = first_mover_of(a.seed_lo, a.seed_hi, g, a.first_mover);
            status = kRunning;
        }
    }
    const Philox r = philox4x32_10(a.seed_lo, a.seed_hi, (uint32_t)ply, (uint32_t)g, (uint32_t)(g >> 32), 0u);
    const int d1 = die_of(r.x[0]), d2 = die_of(r.x[1]);
    const int tail = lane == 28 ? mover : lane == 29 ? d1 : lane == 30 ? d2 : status;
    a.next[q * 32 + lane] = (int8_t)(lane < 28 ? v : tail);
    if (lane == 0) {
        if (a.winner) a.winner[q] = (int8_t)win;
        if (a.ply_out) a.ply_out[q] = ply;
        if (a.gid_out) a.gid_out[q] = (long long)g;
    }
    if (a.next_region) {
        // a finished game that the CALLER restarts will be an opening position: mid-sized
        const int b = status == kRunning ? order_bucket(lane < 28 ? v : 0, lane, mover, d1, d2) : 6;
        if (lane == 0) a.next_region[(size_t)b * n + atomicAdd(&a.next_totals[b], 1u)] = (int32_t)q;
    }
}

// when the CTA of a published double helps before claiming new queue work (bgx_ply.cuh ShareCtx)
struct SelectTune {
    unsigned long long urgent_from;      // queue position from which doubles with >= urgent_min root origins are urgent
    int urgent_min, giant_min;           // giant_min: urgent wherever they sit
};

template <int kWarps, int kSets, bool kExplore>
__global__ void __launch_bounds__(kWarps * 32, 1)
k_select(const int8_t *__restrict__ queries, long long n, float epsilon, uint32_t seed_lo, uint32_t seed_hi,
         SelectOut out, const int32_t *__restrict__ Ti, const float *__restrict__ flat,
         unsigned long long *counter, StealResult *__restrict__ steal, SelectTune tune,
         const int32_t *__restrict__ region, const uint32_t *__restrict__ totals, AdvanceOut adv)
{
    extern __shared__ __align__(128) unsigned char smem[];
    const PlySmem<kWarps, kSets> sm(smem);
    const int lane = threadIdx.x & 31, warp = warp_index();
    PlyCache<kSets> cache;
    cache.reset(sm.scratch[warp].cache, reinterpret_cast<const int4 *>(sm.table), lane);
    sm.init_share();
    stage_table(sm.table, Ti, sm.bar, kFixedBytes);
    PlyEvaluator ev;
    ev.T4 = reinterpret_cast<const int4 *>(sm.table);
    StealResult *cta_results = steal + (size_t)blockIdx.x * kWarps * kStealMaxResults;
    const ShareCtx mine = {&sm.share->slot[warp], cta_results + warp * kStealMaxResults, &sm.share->urgent, 1u << warp,
                           counter, tune.urgent_from, tune.urgent_min, tune.giant_min};
    bool helping = false, first = true;
    const long long first_wave = (long long)gridDim.x * kWarps;
    // sorted queue (k_select_order): lane r < 16 knows where the r-th heaviest bucket ends
    uint32_t bucket_end = 0;
    if (region) {
        bucket_end = lane < kOrderBuckets ? totals[kOrderBuckets - 1 - lane] : 0u;
#pragma unroll
        for (int o = 1; o < kOrderBuckets; o <<= 1) {
            const uint32_t up = __shfl_up_sync(kFull, bucket_end, o);
            if (lane >= o) bucket_end += up;
        }
    }
    for (;;) {
        int root = 0, player = 0, d1 = 0, d2 = 0, vw = 0;
        uint32_t only = 0, u = 0;
        long long q = 0;
        bool explore = false;
        // a sub-tree of a neighbour's double: whenever the queue is empty, and before new queue work if it is a huge one
        if (helping || *(volatile uint32_t *)&sm.share->urgent != 0) {
            bool done;
            only = take_child<kWarps>(sm.share, lane, vw, root, player, d1, done, !helping);
            d2 = d1;
            if (helping && only == 0) {
                if (done) break;
                continue;
            }
        }
        if (only == 0) {
            // the first wave is dealt round-robin over the CTAs (neighbouring queue entries land on different SMs:
            // a run of big doubles must not end up in one CTA, help is intra-CTA); after that, first come first served
            q = first ? (long long)warp * gridDim.x + blockIdx.x : first_wave + claim(counter, lane);
            first = false;
            if (q >= n) {                                   // queue empty: help the owners of big doubles
                helping = true;
                if (lane == 0) atomicSub(&sm.share->active, 1);
                __syncwarp();                               // reconverged before the back-edge (see k_selfplay)
                continue;
            }
            if (region) {                                   // position in the sorted queue -> query
                const int r = __popc(__ballot_sync(kFull, lane < kOrderBuckets && (uint32_t)q >= bucket_end));
                const uint32_t before = __shfl_sync(kFull, bucket_end, r > 0 ? r - 1 : 0);
                q = region[(size_t)(kOrderBuckets - 1 - r) * n + ((uint32_t)q - (r > 0 ? before : 0u))];
            }
            const int b = load_record_byte(queries + q * 32, lane);
            root = lane < 28 ? b : 0;
            player = __shfl_sync(kFull, b, 28) ? 1 : 0; d1 = __shfl_sync(kFull, b, 29); d2 = __shfl_sync(kFull, b, 30);
            if (kExplore && epsilon > 0.f) {
                const Philox r = philox4x32_10(seed_lo, seed_hi, 0u, (uint32_t)q, (uint32_t)((unsigned long long)q >> 32), 2u);
                explore = (float)r.x[0] * 2.3283064365386963e-10f < epsilon;
                u = r.x[1];
            }
        }
        d1 = __shfl_sync(kFull, d1, 0); d2 = __shfl_sync(kFull, d2, 0);        // provably warp-uniform (see k_selfplay)
        player = __shfl_sync(kFull, player, 0); only = __shfl_sync(kFull, only, 0);
        const Choice c = choose_ply_fast<kSets, kExplore>(root, lane, player, d1, d2, ev, cache, explore, u, only ? only : kFull,
                                                          only ? nullptr : &mine);
        if (only) deliver_child<kWarps>(sm.share, cta_results, vw, only, c, lane);
        else {
            store_choice(out, q, c, lane, player);
            if (adv.next) store_advanced(adv, q, n, c.v, lane, player);
        }
        __syncwarp();                                       // reconverged before the back-edge (see k_selfplay)
    }
}

// ---- the rest of a host-driven ply: game over? flip the mover, roll the next dice ---------------
__global__ void k_advance(const int8_t *chosen, int8_t *next, long long n, uint32_t seed_lo,
                          uint32_t seed_hi, int ply, const long long *__restrict__ game_id, int8_t *__restrict__ winner,
                          const int32_t *__restrict__ ply_of = nullptr)
{
    const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
    const int lane = threadIdx.x & 31;
    for (long long q = (long long)blockIdx.x * (blockDim.x >> 5) + warp_index(); q < n; q += warps) {
        const int b = load_record_byte(chosen + q * 32, lane);
        const int off1 = __shfl_sync(kFull, b, 26), off2 = __shfl_sync(kFull, b, 27), mover = __shfl_sync(kFull, b, 28) ? 1 : 0;
        const int win = off1 == 15 ? 0 : (off2 == 15 ? 1 : -1);            // game.cpp:388-407
        const unsigned long long g = game_id ? (unsigned long long)game_id[q] : (unsigned long long)q;
        const Philox r = philox4x32_10(seed_lo, seed_hi, (uint32_t)(ply_of ? ply_of[q] : ply), (uint32_t)g, (uint32_t)(g >> 32), 0u);
        const int tail = lane == 28 ? (win < 0 ? mover ^ 1 : mover) : lane == 29 ? die_of(r.x[0]) : lane == 30 ? die_of(r.x[1]) : win + 1;
        next[q * 32 + lane] = (int8_t)(lane < 28 ? b : tail);
        if (winner && lane == 0) winner[q] = (int8_t)win;
    }
}

// ---- self-play population: play_game (train.py:64-121) for n_slots games at once ---------
struct SelfplayParams {
    int8_t *slots;          // [n_slots][32]: position, byte 28 player to move, byte 31 status
    int32_t *ply;           // [n_slots] plies played in the current game
    long long *game_id;     // [n_slots]
    int8_t *traj_pre;       // [n_slots][traj_cap][32] pre-move records (bytes 29,30 = dice) or NULL
    int8_t *traj_chosen;    // [n_slots][traj_cap][32] chosen afterstates or NULL
    long long n_slots, id_stride;
    uint32_t seed_lo, seed_hi;
    int first_mover, traj_cap;
    int n_plies;            // step mode: plies per slot per call
    int round_mode;         // 1: play the current game to its end, no restart
    float epsilon;
    unsigned long long *counter;
    unsigned long long *stats;   // plies, sequences, scored, finished, p1 wins, truncated, (td steps), tree edges
    int4 *zstash;                // [CTA][warp][32]: per lane, the hidden pre-activation of the warp's best afterstate (greedy_ply)
};

template <int kWarps, int kSets, bool kExplore>
__global__ void __launch_bounds__(kWarps * 32, 1)
k_selfplay(SelfplayParams p, const int32_t *__restrict__ Ti, const float *__restrict__ flat, StealResult *__restrict__ steal)
{
    extern __shared__ __align__(128) unsigned char smem[];
    const PlySmem<kWarps, kSets> sm(smem);
    const int lane = threadIdx.x & 31, warp = warp_index();
    PlyCache<kSets> cache;
    cache.reset(sm.scratch[warp].cache, reinterpret_cast<const int4 *>(sm.table), lane);
    sm.init_share();
    stage_table(sm.table, Ti, sm.bar, kFixedBytes);
    PlyEvaluator ev;
    ev.T4 = reinterpret_cast<const int4 *>(sm.table);
    StealResult *cta_results = steal + (size_t)blockIdx.x * kWarps * kStealMaxResults;
    const ShareCtx mine = {&sm.share->slot[warp], cta_results + warp * kStealMaxResults, &sm.share->urgent, 1u << warp,
                           p.counter, (unsigned long long)(p.n_slots - p.n_slots / 4), 8, kGiantMinChildren};

    unsigned long long *cta_stats = sm.share->stats;    // plies, sequences, scored, finished, p1 wins, truncated, -, tree edges
    const int budget = p.round_mode ? 0x7fffffff : p.n_plies;
    bool helping = false, seated = false;
    int v = 0, dice = 0;                                // dice: d1 | d2 << 4 of one of the game's next plies (WarpSeat::dice_base)
    WarpSeat &S = sm.seat[warp];
    int4 *const zmine = p.zstash + ((size_t)blockIdx.x * kWarps + warp) * 32 + lane;
    // one iteration = one ply: of the slot this warp is seated at, or of a sub-tree taken from a neighbour
    // (whenever the queue is empty, and before its own next ply if the neighbour's double is a huge one)
    for (;;) {
        int root = 0, mover = 0, d1 = 0, d2 = 0, vw = 0;
        uint32_t only = 0, u = 0;
        bool explore = false, rec_traj = false;
        if (helping || *(volatile uint32_t *)&sm.share->urgent != 0) {
            bool done;
            only = take_child<kWarps>(sm.share, lane, vw, root, mover, d1, done, !helping);
            d2 = d1;
            if (helping && only == 0) {
                if (done) break;
                continue;
            }
        }
        if (only == 0) {
            if (!seated) {
                const long long slot = claim(p.counter, lane);
                if (slot >= p.n_slots) {
                    helping = true;
                    if (lane == 0) atomicSub(&sm.share->active, 1);
                    __syncwarp();                                // (see the end of the loop body)
                    continue;
                }
                const int b = load_record_byte(p.slots + slot * 32, lane);
                v = lane < 28 ? b : 0;
                const int status = __shfl_sync(kFull, b, 31);
                if (p.round_mode && status != kRunning) continue;
                const int mover0 = __shfl_sync(kFull, b, 28) ? 1 : 0;
                if (lane == 0) {
                    S.slot = slot;
                    S.player = mover0;
                    S.status = status;
                    S.ply = p.ply[slot];
                    S.gid = (unsigned long long)p.game_id[slot];
                    S.step = 0;
                    S.carry = 0;
                    S.dice_base = -1;
                }
                __syncwarp();
                seated = true;
            }
            const int ply = S.ply;
            if (p.round_mode && p.traj_cap > 0 && ply >= p.traj_cap) {   // the log is full: give the game up
                if (lane == 0) S.status = kTruncated;
                __syncwarp();
                if (lane == 0) atomicAdd(cta_stats + 5, 1ull);
                seated = false;
            } else {
                const unsigned long long gid = S.gid;
                // Philox is counter-based: lane l rolls the dice of ply + l, one evaluation per 32 plies of a game instead of one per ply
                int ahead = ply - S.dice_base;
                if (S.dice_base < 0 || ahead < 0 || ahead >= 32) {
                    const Philox r = philox4x32_10(p.seed_lo, p.seed_hi, (uint32_t)(ply + lane), (uint32_t)gid, (uint32_t)(gid >> 32), 0u);
                    dice = die_of(r.x[0]) | (die_of(r.x[1]) << 4);
                    __syncwarp();
                    if (lane == 0) S.dice_base = ply;
                    __syncwarp();
                    ahead = 0;
                }
                const int rolled = __shfl_sync(kFull, dice, ahead);
                d1 = rolled & 15; d2 = rolled >> 4;
                mover = S.player;
                rec_traj = p.traj_pre != nullptr && ply < p.traj_cap && S.status == kRunning;
                if (rec_traj) {
                    int8_t *t = p.traj_pre + ((size_t)S.slot * p.traj_cap + ply) * 32;
                    const int out = lane < 28 ? v : (lane == 28 ? mover : (lane == 29 ? d1 : (lane == 30 ? d2 : 0)));
                    t[lane] = (int8_t)out;                           // train.py:105-106
                }
                if (kExplore && p.epsilon > 0.f) {
                    const Philox e = philox4x32_10(p.seed_lo, p.seed_hi, (uint32_t)ply, (uint32_t)gid, (uint32_t)(gid >> 32), 2u);
                    explore = (float)e.x[0] * 2.3283064365386963e-10f < p.epsilon;
                    u = e.x[1];
                }
                root = v;
            }
        }
        if (only || seated) {
            // what the walk branches on, as values ptxas can PROVE warp-uniform (shuffles from a fixed lane): with dice or a mover
            // that merely happen to be uniform every loop of the walk counts as divergent and each *_sync intrinsic in it is
            // guarded by BRA.DIV + reconvergence code
            d1 = __shfl_sync(kFull, d1, 0); d2 = __shfl_sync(kFull, d2, 0);
            mover = __shfl_sync(kFull, mover, 0); only = __shfl_sync(kFull, only, 0);
            const Choice c = choose_ply_fast<kSets, kExplore>(root, lane, mover, d1, d2, ev, cache, explore, u, only ? only : kFull,
                                                              only ? nullptr : &mine, only ? nullptr : zmine,
                                                              only == 0 && S.carry != 0);              // model.py:180-222
            if (only) {
                deliver_child<kWarps>(sm.share, cta_results, vw, only, c, lane);
                continue;
            }
            v = c.v;
            if (lane == 0) {
                atomicAdd(cta_stats + 0, 1ull);
                atomicAdd(cta_stats + 1, (unsigned long long)c.n_seq);
                atomicAdd(cta_stats + 2, (unsigned long long)c.n_scored);
                atomicAdd(cta_stats + 7, (unsigned long long)c.n_visited);
            }
            if (rec_traj && p.traj_chosen) {
                int8_t *t = p.traj_chosen + ((size_t)S.slot * p.traj_cap + S.ply) * 32;
                const int len = (int)(c.moves >> 40);
                const int out = lane < 28 ? v : (lane == 28 ? S.player : (lane == 31 ? (len > 0 ? 1 : 0) : 0));
                t[lane] = (int8_t)out;
            }
            // is_game_over (game.cpp:388-407): PLAYER1 is checked first
            const int off1 = __shfl_sync(kFull, v, 26), off2 = __shfl_sync(kFull, v, 27);
            const int winner = off1 == 15 ? 0 : (off2 == 15 ? 1 : -1);
            const int step = S.step + 1;
            const int mover_now = S.player;
            unsigned long long gid = S.gid;
            int next_player = mover_now ^ 1, next_ply = S.ply + 1, next_status = kRunning;   // train.py:119-120
            if (winner >= 0) {
                if (lane == 0) {
                    atomicAdd(cta_stats + 3, 1ull);
                    if (winner == 0) atomicAdd(cta_stats + 4, 1ull);
                }
                if (p.round_mode) {
                    next_status = winner == 0 ? kP1Won : kP2Won;
                    next_player = mover_now;
                    seated = false;
                } else {
                    gid += (unsigned long long)p.id_stride;          // restart in place
                    v = start_value(lane);
                    next_player = first_mover_of(p.seed_lo, p.seed_hi, gid, p.first_mover);
                    next_ply = 0;
                }
            }
            __syncwarp();
            if (lane == 0) { S.step = step; S.player = next_player; S.ply = next_ply; S.status = next_status; S.gid = gid; S.carry = c.z_ok && winner < 0; if (winner >= 0) S.dice_base = -1; }
            __syncwarp();
            if (step >= budget) seated = false;
        }
        if (!seated) {                                               // leave the slot: write it back
            const long long slot = S.slot;
            const int out = lane < 28 ? v : (lane == 28 ? S.player : (lane == 31 ? S.status : 0));
            p.slots[slot * 32 + lane] = (int8_t)out;
            if (lane == 0) {
                p.ply[slot] = S.ply;
                p.game_id[slot] = (long long)S.gid;
            }
        }
        // Reconverge before the back-edge: a lane-0 block that ends an iteration lets the other lanes reach the loop header
        // first, ptxas then treats the WHOLE loop body as possibly diverged and guards every *_sync intrinsic in it - the
        // walk included - with BRA.DIV + reconvergence code (47 sites, ~10 % of the executed instructions).
        __syncwarp();
    }
    // the last warp to leave flushes the CTA's statistics
    __syncwarp();
    __threadfence_block();
    int last = 0;
    if (lane == 0) last = atomicAdd(&sm.share->pad[0], 1) == kWarps - 1;
    if (__shfl_sync(kFull, last, 0) && lane < 8 && lane != 6) atomicAdd(p.stats + lane, cta_stats[lane]);
}

// ---- are the SFU approximations the ply evaluator ranks by monotone?  (PlyEvaluator::value_of) ----------------
// The greedy ply compares integer output sums and evaluates V = 1 / (1 + 2^a) only for a sum that beats the best so far.
// That equals comparing V itself if V is a non-decreasing function of the sum: the FFMA, the multiply and the add are
// correctly rounded, hence monotone; ex2.approx.ftz and rcp.approx.ftz are table-based approximations with no such
// guarantee on paper.  This kernel checks them on the device, exhaustively: every pair of neighbouring finite floats for
// ex2, every pair of neighbours in [1, FLT_MAX] for rcp (its argument is 1 + 2^a >= 1).  out[0] / out[1]: violations.
__device__ __forceinline__ float ordered_float(uint32_t k)            // k ascending <=> value ascending (k >= 2^31: positive)
{
    return __uint_as_float(k & 0x80000000u ? k ^ 0x80000000u : ~k);
}
__global__ void k_sfu_monotone(unsigned long long *out)
{
    unsigned long long bad_ex2 = 0, bad_rcp = 0;
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long k = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; k < 0xFFFFFFFFull; k += stride) {
        const float a = ordered_float((uint32_t)k), b = ordered_float((uint32_t)k + 1u);
        if (!(fabsf(a) <= 3.402823466e38f) || !(fabsf(b) <= 3.402823466e38f)) continue;       // NaN / infinity
        float ea, eb;
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(ea) : "f"(a));
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(eb) : "f"(b));
        if (!(ea <= eb)) bad_ex2++;
        if (a >= 1.0f) {
            float ra, rb;
            asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(ra) : "f"(a));
            asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rb) : "f"(b));
            if (!(ra >= rb)) bad_rcp++;
        }
    }
    if (bad_ex2) atomicAdd(out + 0, bad_ex2);
    if (bad_rcp) atomicAdd(out + 1, bad_rcp);
}

// (re)seat every slot: opening position, first mover, ply 0
__global__ void k_selfplay_reset(int8_t *slots, int32_t *ply, long long *game_id, long long n_slots,
                                 long long first_id, long long id_stride, int advance,
                                 uint32_t seed_lo, uint32_t seed_hi, int first_mover)
{
    const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
    const int lane = threadIdx.x & 31;
    for (long long s = (long long)blockIdx.x * (blockDim.x >> 5) + warp_index(); s < n_slots; s += warps) {
        const unsigned long long gid = advance ? (unsigned long long)(game_id[s] + id_stride) : (unsigned long long)(first_id + s);
        const int player = first_mover_of(seed_lo, seed_hi, gid, first_mover);
        const int out = lane < 28 ? start_value(lane) : (lane == 28 ? player : 0);
        slots[s * 32 + lane] = (int8_t)out;
        if (lane == 0) { ply[s] = 0; game_id[s] = (long long)gid; }
    }
}

// `per_game` recorded pre-move records of every slot's current game, each at a uniformly drawn ply (Philox stream 3):
// the playout half of the enumeration sweep (BASELINE.json configs[1], SURVEY.md 8d config 2)
__global__ void k_traj_sample(const int8_t *__restrict__ traj, const int32_t *__restrict__ ply, long long n_slots, int traj_cap,
                              int per_game, uint32_t seed_lo, uint32_t seed_hi, int8_t *__restrict__ out)
{
    const long long warps = (long long)gridDim.x * (blockDim.x >> 5), total = n_slots * per_game;
    const int lane = threadIdx.x & 31;
    for (long long i = (long long)blockIdx.x * (blockDim.x >> 5) + warp_index(); i < total; i += warps) {
        const long long slot = i / per_game;
        const int j = (int)(i % per_game);
        int T = ply[slot];
        if (T > traj_cap) T = traj_cap;
        int b = 0;
        if (T > 0) {
            const Philox r = philox4x32_10(seed_lo, seed_hi, (uint32_t)j, (uint32_t)slot, (uint32_t)((unsigned long long)slot >> 32), 3u);
            const int t = (int)mulhi32(r.x[0], (uint32_t)T);
            b = load_record_byte(traj + ((size_t)slot * traj_cap + t) * 32, lane);
        }
        out[i * 32 + lane] = (int8_t)(lane == 31 ? 0 : b);
    }
}

} // namespace bgx
