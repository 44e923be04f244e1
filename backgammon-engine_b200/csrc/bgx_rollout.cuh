// bgx_rollout.cuh — rollouts (DESIGN 7d): Monte Carlo evaluation of arbitrary positions under the net's greedy one-ply policy.
//   k_rollout          persistent, one warp per trial at a time: claims work item i = position x trials + trial, plays the trial
//                      from the position to its end or its truncation ply with the fused greedy ply (choose_ply_fast, the root-stash
//                      carry, big doubles shared inside the CTA) and writes x_t, the outcome class and the ply count at index i
//   k_rollout_reduce   one thread per position: mean, standard error and counts, float64, sequentially in trial order
// Dice are a function of the trial index only (common random numbers), the values are the fixed-point evaluator's (pure functions
// of the query, bgx_ply.cuh) and every trial's result lands at its own index: the outputs depend on nothing but
// (position, mover, trials, max_plies, seed, flags, weights).
#pragma once
#include "bgx_kernels.cuh"

namespace bgx {

constexpr int kRolloutStream = 4;        // Philox stream of the rollout dice (0 self-play, 1 roll-off, 2 exploration, 3 sampling)

struct RolloutParams {
    const int8_t *positions;  // [n_pos][32] of this launch: position, byte 28 = player on roll
    long long n_items;        // n_pos x trials
    int trials, cap;          // cap: the truncation ply (max_plies, or BGX_ROLLOUT_MAX_PLIES for "play to the end")
    int stratify;             // ply 0 of trial t rolls t mod 36
    uint32_t seed_lo, seed_hi;
    float *value;             // [n_items] x_t
    int8_t *outcome;          // [n_items] 0 truncated, 1..3 PLAYER1 single / gammon / backgammon, 4..6 PLAYER2
    int32_t *plies;           // [n_items]
    unsigned long long *counter;
    int4 *zstash;             // [CTA][warp][32] (greedy_ply's root-stash carry)
};

// outcome class of a finished game, from the final board alone.  The loser is gammoned if it has borne nothing off, backgammoned
// if it also has a checker on the bar or in the winner's home board (PLAYER1 bears off past index 23: its home is 18..23,
// PLAYER2's is 0..5; bars are lanes 24 + player, counts positive, PLAYER1's checkers positive on the points)
__device__ __forceinline__ int outcome_class(int v, int lane, int winner)
{
    const int loser_off = __shfl_sync(kFull, v, 27 - winner);
    const int loser_bar = __shfl_sync(kFull, v, 25 - winner);
    const bool in_home = winner == 0 ? (lane >= 18 && lane < 24 && v < 0) : (lane < 6 && v > 0);
    const bool back = loser_bar != 0 || __ballot_sync(kFull, in_home) != 0;
    const int cls = loser_off != 0 ? 1 : (back ? 3 : 2);
    return winner == 0 ? cls : 3 + cls;
}

template <int kWarps, int kSets>
__global__ void __launch_bounds__(kWarps * 32, 1)
k_rollout(RolloutParams p, const int32_t *__restrict__ Ti, StealResult *__restrict__ steal)
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
                           p.counter, (unsigned long long)(p.n_items - p.n_items / 4), 8, kGiantMinChildren};
    bool helping = false, seated = false;
    int v = 0, dice = 0;                                // dice: d1 | d2 << 4 of ply dice_base + lane of the trial
    WarpSeat &S = sm.seat[warp];                        // slot = work item, gid = trial index, ply = plies played so far
    int4 *const zmine = p.zstash + ((size_t)blockIdx.x * kWarps + warp) * 32 + lane;
    // one iteration = one ply: of the trial this warp is seated at, or of a sub-tree taken from a neighbour (k_selfplay's loop)
    for (;;) {
        int root = 0, mover = 0, d1 = 0, d2 = 0, vw = 0;
        uint32_t only = 0;
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
                const long long i = claim(p.counter, lane);
                if (i >= p.n_items) {
                    helping = true;
                    if (lane == 0) atomicSub(&sm.share->active, 1);
                    __syncwarp();                                // (see the end of the loop body)
                    continue;
                }
                const long long pos = i / p.trials, t = i - pos * p.trials;
                const int b = load_record_byte(p.positions + pos * 32, lane);
                v = lane < 28 ? b : 0;
                const int off1 = __shfl_sync(kFull, v, 26), off2 = __shfl_sync(kFull, v, 27);
                if (off1 == 15 || off2 == 15) {                  // over already: every trial ends at ply 0 (PLAYER1 checked first)
                    const int winner = off1 == 15 ? 0 : 1;
                    const int cls = outcome_class(v, lane, winner);
                    if (lane == 0) { p.value[i] = winner == 0 ? 1.f : 0.f; p.outcome[i] = (int8_t)cls; p.plies[i] = 0; }
                    __syncwarp();
                    continue;
                }
                const int mover0 = __shfl_sync(kFull, b, 28) ? 1 : 0;
                if (lane == 0) {
                    S.slot = i;
                    S.gid = (unsigned long long)t;
                    S.player = mover0;
                    S.ply = 0;
                    S.carry = 0;
                    S.dice_base = -1;
                }
                __syncwarp();
                seated = true;
            }
            const int ply = S.ply;
            const unsigned long long t = S.gid;
            // Philox is counter-based: lane l rolls the dice of ply + l, one evaluation per 32 plies of a trial
            int ahead = ply - S.dice_base;
            if (S.dice_base < 0 || ahead >= 32) {
                const Philox r = philox4x32_10(p.seed_lo, p.seed_hi, (uint32_t)(ply + lane), (uint32_t)t, (uint32_t)(t >> 32),
                                               (uint32_t)kRolloutStream);
                dice = die_of(r.x[0]) | (die_of(r.x[1]) << 4);
                __syncwarp();
                if (lane == 0) S.dice_base = ply;
                __syncwarp();
                ahead = 0;
            }
            const int rolled = __shfl_sync(kFull, dice, ahead);
            d1 = rolled & 15; d2 = rolled >> 4;
            if (p.stratify && ply == 0) {                        // stratified first roll: each ordered roll trials / 36 times
                const int r = (int)(t % 36u);
                d1 = 1 + r / 6; d2 = 1 + r % 6;
            }
            mover = S.player;
            root = v;
        }
        // what the walk branches on, as values ptxas can PROVE warp-uniform (see k_selfplay)
        d1 = __shfl_sync(kFull, d1, 0); d2 = __shfl_sync(kFull, d2, 0);
        mover = __shfl_sync(kFull, mover, 0); only = __shfl_sync(kFull, only, 0);
        const Choice c = choose_ply_fast<kSets, false>(root, lane, mover, d1, d2, ev, cache, false, 0u, only ? only : kFull,
                                                       only ? nullptr : &mine, only ? nullptr : zmine,
                                                       only == 0 && S.carry != 0);
        if (only) {
            deliver_child<kWarps>(sm.share, cta_results, vw, only, c, lane);
            continue;
        }
        v = c.v;
        const int off1 = __shfl_sync(kFull, v, 26), off2 = __shfl_sync(kFull, v, 27);
        const int winner = off1 == 15 ? 0 : (off2 == 15 ? 1 : -1);          // game.cpp:388-407
        const int played = S.ply + 1;
        const bool cut = winner < 0 && played >= p.cap;
        if (winner >= 0 || cut) {
            float x;
            int cls = 0;
            if (winner >= 0) {
                x = winner == 0 ? 1.f : 0.f;
                cls = outcome_class(v, lane, winner);
            } else {
                // the value the truncation ply reports; without a sequence (or with only the empty one of a blocked double) the
                // position itself for its mover, from scratch (k_twoply_reduce's rule for a blocked reply)
                x = c.value;
                if (!c.any) x = ev.finish(ev.preactivation(root, lane, mover), lane);
            }
            const long long i = S.slot;
            if (lane == 0) { p.value[i] = x; p.outcome[i] = (int8_t)cls; p.plies[i] = played; }
            seated = false;
        }
        __syncwarp();
        if (lane == 0) { S.ply = played; S.player = S.player ^ 1; S.carry = c.z_ok && winner < 0; }
        // Reconverge before the back-edge (see k_selfplay): otherwise every *_sync intrinsic of the walk is guarded by BRA.DIV
        __syncwarp();
    }
}

// per position: mean and standard error of x_t, float64, each sum in trial order (d * d rounded before it is added: no FMA
// contraction, so the result is the plain sequential sum), and the counts of the outcome classes 1..6, of truncated trials and
// of plies
__global__ void k_rollout_reduce(const float *__restrict__ value, const int8_t *__restrict__ outcome, const int32_t *__restrict__ plies,
                                 long long n_pos, int trials, double *mean, double *std_err, long long *counts)
{
    const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n_pos) return;
    const float *x = value + q * trials;
    double sum = 0.0;
    for (int t = 0; t < trials; t++) sum = __dadd_rn(sum, (double)x[t]);
    const double m = sum / (double)trials;
    if (mean) mean[q] = m;
    if (std_err) {
        double ss = 0.0;
        for (int t = 0; t < trials; t++) {
            const double d = __dadd_rn((double)x[t], -m);
            ss = __dadd_rn(ss, __dmul_rn(d, d));
        }
        std_err[q] = trials > 1 ? sqrt(ss / ((double)trials * (double)(trials - 1))) : __longlong_as_double(0x7ff8000000000000ll);
    }
    if (counts) {
        long long c[8] = {};
        for (int t = 0; t < trials; t++) {
            const int k = outcome[q * trials + t];
            c[k == 0 ? 6 : k - 1]++;
            c[7] += plies[q * trials + t];
        }
        for (int k = 0; k < 8; k++) counts[q * 8 + k] = c[k];
    }
}

} // namespace bgx
