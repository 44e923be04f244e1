// bgx_twoply.cuh — two-ply move selection (DESIGN 7c): the mover's distinct afterstates, each valued by the expectation over
// the opponent's 21 rolls of the opponent's own greedy reply.  The replies are ordinary one-ply queries and go through k_select
// unchanged; the kernels here only build its input and reduce its output:
//   k_candidates      one warp per query: the distinct afterstates in first-appearance order (the summary kernel's leaf and
//                     exact-dedup table), each with its first sequence and its one-ply value
//   k_twoply_expand   one warp per query: win detection and the top-K filter; k_twoply_list compacts the expanded candidates
//   k_twoply_replies  21 reply records per expanded candidate of a chunk
//   k_twoply_reduce   one warp per expanded candidate: the fp64 expectation in roll order
//   k_twoply_pick     one warp per query: the pick, written as store_choice writes a one-ply choice
// Every value is a pure function of (query, weights, K): candidate order is the reference's enumeration order, the one-ply and
// reply values are the fixed-point evaluator's (bgx_ply.cuh), and the sums run in a fixed order.
#pragma once
#include "bgx_kernels.cuh"

namespace bgx {

// the opponent's rolls in the fixed order a = 1..6, b = 1..a; a roll with a != b stands for both orders (weight 2 of 36)
constexpr int kRolls = 21;
__device__ __constant__ int8_t kRollA[kRolls] = {1, 2, 2, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 5, 6, 6, 6, 6, 6, 6};
__device__ __constant__ int8_t kRollB[kRolls] = {1, 1, 2, 1, 2, 3, 1, 2, 3, 4, 1, 2, 3, 4, 5, 1, 2, 3, 4, 5, 6};

// a candidate bears off the mover's 15th checker: the game is won
__device__ __forceinline__ bool wins(const int8_t *rec, int player) { return rec[26 + player] == 15; }

// counts of the candidate lists: U of the summary walk, -1 (table overflow) counted as 0 and reported in flags[0]
__global__ void k_twoply_count(const int32_t *__restrict__ n_unique, long long n, int32_t *__restrict__ count, int *flags)
{
    const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n) return;
    const int u = n_unique[q];
    count[q] = u < 0 ? 0 : u;
    if (u < 0) atomicOr(flags, 1);
}

// writes every distinct afterstate once, at its first appearance in reference order: record (byte 28 = mover), first sequence,
// one-ply value V(s, mover) of the fixed-point evaluator (what k_select compares).  The summary walk's leaf does the exact dedup
// (a new afterstate is one that raised its U), so both walks agree on U by construction.
struct CandidateLeaf {
    SummaryLeaf seen;
    int player;
    const PlyEvaluator *ev;
    int8_t *rec, *moves, *lens;      // this query's first row
    float *val;
    int cap;                         // rows reserved for the query (its U)

    __device__ __forceinline__ void operator()(int v, uint64_t mv, int len)
    {
        const int n = seen.n_unique;
        seen(v, mv, len);
        if (seen.n_unique == n) return;
        const int lane = seen.lane;
        if (n < cap) {
            rec[n * 32 + lane] = (int8_t)(lane < 28 ? v : (lane == 28 ? player : 0));
            if (lane < 8) {
                const int j = lane >> 1;
                const int code = (int)((mv >> (10 * j + 5 * (lane & 1))) & 31u);
                moves[n * 8 + lane] = (int8_t)(j < len ? code : 0);
            }
            if (lane == 8) lens[n] = (int8_t)len;
            const float V = ev->finish(ev->preactivation(v, lane, player), lane);
            if (lane == 0) val[n] = V;
        }
        __syncwarp();
    }
};

__global__ void __launch_bounds__(kGameThreads, 1)
k_candidates(const int8_t *__restrict__ queries, long long n, const int32_t *__restrict__ count, const long long *__restrict__ offsets,
             int8_t *__restrict__ rec, int8_t *__restrict__ moves, int8_t *__restrict__ lens, float *__restrict__ val,
             uint32_t *__restrict__ tables, uint32_t *__restrict__ gens, unsigned long long *counter, int *flags,
             const int32_t *__restrict__ Ti)
{
    extern __shared__ __align__(128) unsigned char smem[];
    int32_t *sT = reinterpret_cast<int32_t *>(smem);
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem + kFixedBytes);
    stage_table(sT, Ti, bar, kFixedBytes);
    PlyEvaluator ev;
    ev.T4 = reinterpret_cast<const int4 *>(sT);
    const int lane = threadIdx.x & 31;
    const int gwarp = blockIdx.x * (blockDim.x >> 5) + warp_index();
    uint32_t *table = tables + (size_t)gwarp * (kUniqBytesPerWarp / 4);
    uint32_t gen = gens[gwarp];
    for (;;) {
        const long long q = claim(counter, lane);
        if (q >= n) break;
        const int b = load_record_byte(queries + q * 32, lane);
        const int root = lane < 28 ? b : 0;
        const int player = __shfl_sync(kFull, b, 28) ? 1 : 0, d1 = __shfl_sync(kFull, b, 29), d2 = __shfl_sync(kFull, b, 30);
        gen = (gen + 1) & 0xFFu;                    // (as k_enumerate_summary: the tables and generations are shared)
        if (gen == 0) {
            for (int i = lane; i < kUniqSlots * kUniqWords; i += 32) table[i] = 0;
            gen = 1;
            __syncwarp();
        }
        const long long base = offsets[q];
        CandidateLeaf leaf;
        leaf.seen.table = table; leaf.seen.gen = gen; leaf.seen.lane = lane; leaf.player = player; leaf.ev = &ev;
        leaf.rec = rec + base * 32; leaf.moves = moves + base * 8; leaf.lens = lens + base; leaf.val = val + base;
        leaf.cap = count[q];
        walk_turn(root, lane, player, d1, d2, leaf);
        if (lane == 0 && (leaf.seen.overflow || leaf.seen.n_unique != leaf.cap)) atomicOr(flags, 2);      // never seen: the summary walk sized it
        __syncwarp();                               // reconverged before the back-edge (see k_selfplay)
    }
    if (lane == 0) gens[gwarp] = gen;
}

// which candidates are expanded: none if one of them wins, else all (K = 0 or K >= U) or the K best by one-ply value (signed for
// the mover, first appearance on ties: with K = 1 that is k_select's own pick)
__global__ void k_twoply_expand(const int8_t *__restrict__ queries, long long n, const int32_t *__restrict__ count,
                                const long long *__restrict__ offsets, const int8_t *__restrict__ rec, const float *__restrict__ val,
                                int K, int8_t *__restrict__ expand, int32_t *__restrict__ n_exp)
{
    const int lane = threadIdx.x & 31;
    const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
    for (long long q = (long long)blockIdx.x * (blockDim.x >> 5) + warp_index(); q < n; q += warps) {
        const int U = count[q];
        const long long base = offsets[q];
        const int player = queries[q * 32 + 28] ? 1 : 0;
        bool win = false;
        for (int i = lane; i < U; i += 32) win |= wins(rec + (base + i) * 32, player);
        win = __any_sync(kFull, win);
        int total = 0;
        for (int i0 = 0; i0 < U; i0 += 32) {
            const int i = i0 + lane;
            bool e = false;
            if (i < U && !win) {
                if (K == 0 || K >= U) {
                    e = true;
                } else {
                    const float ki = player ? -val[base + i] : val[base + i];
                    int rank = 0;
                    for (int j = 0; j < U && rank < K; j++) {
                        const float kj = player ? -val[base + j] : val[base + j];
                        rank += (kj > ki || (kj == ki && j < i)) ? 1 : 0;
                    }
                    e = rank < K;
                }
            }
            if (i < U) expand[base + i] = e ? 1 : 0;
            total += __popc(__ballot_sync(kFull, e));
        }
        if (lane == 0) n_exp[q] = total;
    }
}

// the expanded candidates of all queries, in query order and first appearance within a query: list[exp_off[q] + r]
__global__ void k_twoply_list(long long n, const int32_t *__restrict__ count, const long long *__restrict__ offsets,
                              const int8_t *__restrict__ expand, const long long *__restrict__ exp_off, long long *__restrict__ list)
{
    const int lane = threadIdx.x & 31;
    const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
    for (long long q = (long long)blockIdx.x * (blockDim.x >> 5) + warp_index(); q < n; q += warps) {
        const int U = count[q];
        const long long base = offsets[q];
        long long at = exp_off[q];
        for (int i0 = 0; i0 < U; i0 += 32) {
            const int i = i0 + lane;
            const bool e = i < U && expand[base + i];
            const uint32_t m = __ballot_sync(kFull, e);
            if (e) list[at + __popc(m & ((1u << lane) - 1u))] = base + i;
            at += __popc(m);
        }
    }
}

// reply r of the chunk that starts at expanded candidate e0: candidate list[e0 + r / 21], opponent to move, roll r % 21
__global__ void k_twoply_replies(const long long *__restrict__ list, long long e0, long long n_replies, const int8_t *__restrict__ rec,
                                 int8_t *__restrict__ replies)
{
    const int lane = threadIdx.x & 31;
    const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
    for (long long r = (long long)blockIdx.x * (blockDim.x >> 5) + warp_index(); r < n_replies; r += warps) {
        const long long c = list[e0 + r / kRolls];
        const int roll = (int)(r % kRolls);
        const int b = load_record_byte(rec + c * 32, lane);
        const int opp = __shfl_sync(kFull, b, 28) ^ 1;
        const int out = lane < 28 ? b : lane == 28 ? opp : lane == 29 ? kRollA[roll] : lane == 30 ? kRollB[roll] : 0;
        replies[r * 32 + lane] = (int8_t)out;
    }
}

// E2 of the chunk's expanded candidates: sum over the rolls of weight x reply value, in roll order, in float64, rounded once.
// A reply k_select reports as NaN (the opponent has no sequence) is the position itself: V(A, opponent), k_evaluate's path.
__global__ void __launch_bounds__(kGameThreads, 1)
k_twoply_reduce(const long long *__restrict__ list, long long e0, long long e1, const int8_t *__restrict__ rec,
                const float *__restrict__ reply_value, float *__restrict__ e2, const int32_t *__restrict__ Ti)
{
    extern __shared__ __align__(128) unsigned char smem[];
    int32_t *sT = reinterpret_cast<int32_t *>(smem);
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem + kFixedBytes);
    stage_table(sT, Ti, bar, kFixedBytes);
    PlyEvaluator ev;
    ev.T4 = reinterpret_cast<const int4 *>(sT);
    const int lane = threadIdx.x & 31;
    const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
    for (long long e = e0 + (long long)blockIdx.x * (blockDim.x >> 5) + warp_index(); e < e1; e += warps) {
        const long long c = list[e];
        float R = lane < kRolls ? reply_value[(e - e0) * kRolls + lane] : 0.f;
        const uint32_t blocked = __ballot_sync(kFull, lane < kRolls && R != R);
        if (blocked) {
            const int b = load_record_byte(rec + c * 32, lane);
            const int opp = __shfl_sync(kFull, b, 28) ^ 1;
            const float V = ev.finish(ev.preactivation(lane < 28 ? b : 0, lane, opp), lane);
            if ((blocked >> lane) & 1u) R = V;
        }
        const double term = lane < kRolls ? (kRollA[lane] == kRollB[lane] ? 1.0 : 2.0) * (double)R : 0.0;
        double acc = 0.0;
        for (int r = 0; r < kRolls; r++) acc += __shfl_sync(kFull, term, r);
        if (lane == 0) e2[c] = (float)(acc / 36.0);
    }
}

// the pick of every query: the first winning candidate (value 1 / 0), else the first-appearance arg-max (PLAYER1) / arg-min
// (PLAYER2) of E2 over the expanded candidates; no candidate: the position comes back, value NaN
__global__ void k_twoply_pick(const int8_t *__restrict__ queries, long long n, const int32_t *__restrict__ count,
                              const long long *__restrict__ offsets, const int8_t *__restrict__ rec, const int8_t *__restrict__ cmoves,
                              const int8_t *__restrict__ clens, const int8_t *__restrict__ expand, const float *__restrict__ e2,
                              const int32_t *__restrict__ n_exp, int8_t *chosen, int8_t *moves, int8_t *moves_len, float *value,
                              int32_t *n_candidates, int32_t *n_expanded)
{
    const int lane = threadIdx.x & 31;
    const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
    for (long long q = (long long)blockIdx.x * (blockDim.x >> 5) + warp_index(); q < n; q += warps) {
        const int U = count[q];
        const long long base = offsets[q];
        const int b = load_record_byte(queries + q * 32, lane);
        const int player = __shfl_sync(kFull, b, 28) ? 1 : 0;
        int best = -1;
        float v = __int_as_float(0x7fc00000);
        for (int i0 = 0; i0 < U && best < 0; i0 += 32) {
            const uint32_t m = __ballot_sync(kFull, i0 + lane < U && wins(rec + (base + i0 + lane) * 32, player));
            if (m) {
                best = i0 + lowest_bit(m);
                v = player ? 0.f : 1.f;
            }
        }
        if (best < 0 && U > 0) {
            float key = __int_as_float(0xff800000);         // -inf: signed for the mover, maximised, strict > keeps the first
            int idx = INT_MAX;
            for (int i = lane; i < U; i += 32) {
                if (!expand[base + i]) continue;
                const float x = e2[base + i];
                const float k = player ? -x : x;
                if (k > key) { key = k; idx = i; }
            }
            for (int o = 16; o > 0; o >>= 1) {
                const float k2 = __shfl_xor_sync(kFull, key, o);
                const int i2 = __shfl_xor_sync(kFull, idx, o);
                if (k2 > key || (k2 == key && i2 < idx)) { key = k2; idx = i2; }
            }
            best = idx;
            v = player ? -key : key;
        }
        int len = 0;
        if (best >= 0) {
            const long long c = base + best;
            len = clens[c];
            if (chosen) chosen[q * 32 + lane] = (int8_t)(lane < 31 ? (int)rec[c * 32 + lane] : (len > 0 ? 1 : 0));
            if (moves && lane < 8) moves[q * 8 + lane] = cmoves[c * 8 + lane];
        } else {
            if (chosen) chosen[q * 32 + lane] = (int8_t)(lane < 28 ? b : (lane == 28 ? player : 0));
            if (moves && lane < 8) moves[q * 8 + lane] = 0;
        }
        if (lane == 0) {
            if (moves_len) moves_len[q] = (int8_t)len;
            if (value) value[q] = v;
            if (n_candidates) n_candidates[q] = U;
            if (n_expanded) n_expanded[q] = n_exp[q];
        }
    }
}

} // namespace bgx
