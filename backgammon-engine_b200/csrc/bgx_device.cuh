// bgx_device.cuh — device-side building blocks of the self-play hot path (sm_100a).
//
// Execution model: ONE WARP PER POSITION.  Lane i (0..27) holds element i of the
// reference's 28-int state row (cppsrc/game.hpp:17-28): lanes 0..23 the board points,
// 24/25 the bar counts, 26/27 the borne-off counts; lanes 28..31 hold 0.  Everything a
// rule needs about the whole board is two __ballot_sync masks in the mover's frame (struct
// Mover; the mask algebra is bgx_core.h's), a move is one shuffle and three predicated adds,
// and the turn tree of cppsrc/game.cpp:109-191 is walked with warp-uniform control flow (no
// divergence, no per-thread stacks in memory).  The 198-128-1 network (model.py:63-67) is
// evaluated by the same warp with 4 hidden units per lane against a feature-major weight
// table resident in shared memory (bgx_ply.cuh).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "bgx_core.h"

namespace bgx {

constexpr unsigned kFull = 0xFFFFFFFFu;
constexpr int kFeatures = 198;
constexpr int kHidden = 128;
constexpr int kTableFloats = kFeatures * kHidden;                 // 25 344
constexpr int kTableBytes = kTableFloats * 4;                     // 101 376
constexpr int kFixedRows = kFeatures + 30 + 4;                    // + borne-off step rows, b1, w2, constants, lane constants (bgx_ply.cuh)
constexpr int kFixedInts = kFixedRows * kHidden;                  // 29 696
constexpr int kFixedBytes = kFixedInts * 4;                       // 118 784
constexpr int kRowB1 = kFeatures + 30;                            // round(b1 S)
constexpr int kRowW2 = kFeatures + 31;                            // w2 (fp32 bit patterns)
constexpr int kRowConst = kFeatures + 32;                         // every float4: {S, -log2(e)/S, b2, Y}
constexpr int kRowLane = kFeatures + 33;                          // word l (l < 32): the hash multiplier of lane l (PlyCache);
                                                                  // word 32 + l: the same in PLAYER2's mover frame

// the ply cache's hash multiplier of a lane: odd, and not a polynomial in the lane (moving a checker by the same die from
// different points must not shift the hash by the same amount)
__host__ __device__ constexpr uint32_t ply_hash_multiplier(int lane) { return (0x9E3779B1u * (uint32_t)(2 * lane + 1)) ^ (0x85EBCA77u >> (lane & 7)); }
// ... of a lane of PLAYER2's mover frame (bgx_ply.cuh mover_frame: points negated, 24 <-> 25, 26 <-> 27): a position hashes
// to the same value in either frame, so the ply cache picks the same sets and victims whoever moves
__host__ __device__ constexpr uint32_t ply_hash_multiplier_p2(int lane)
{
    return lane < 24 ? 0u - ply_hash_multiplier(lane) : ply_hash_multiplier(lane < 28 ? lane ^ 1 : lane);
}

// status byte (record byte 31) of a self-play slot
enum { kRunning = 0, kP1Won = 1, kP2Won = 2, kTruncated = 3 };

// The warp's index in its CTA as a value ptxas can PROVE warp-uniform (a shuffle from a fixed lane).  threadIdx.x >> 5 is
// uniform too, but not provably: everything loaded through it (a warp's seat, its cache, its queue position) then counts as
// divergent, every loop over a ballot mask derived from it as a divergent loop, and every *_sync intrinsic inside gets a
// BRA.DIV guard with its reconvergence code (47 sites in k_selfplay, ~10 % of its executed instructions).
__device__ __forceinline__ int warp_index() { return __shfl_sync(0xFFFFFFFFu, (int)(threadIdx.x >> 5), 0); }

// ------------------------------------------------------------------------------------
// lane-distributed state
// ------------------------------------------------------------------------------------

// the five bit-planes of the row: the canonical 160-bit key of a position
__device__ __forceinline__ void key_planes(int v, uint32_t k[5])
{
    const int mag = v < 0 ? -v : v;
    k[0] = __ballot_sync(kFull, mag & 1);
    k[1] = __ballot_sync(kFull, mag & 2);
    k[2] = __ballot_sync(kFull, mag & 4);
    k[3] = __ballot_sync(kFull, mag & 8);
    k[4] = __ballot_sync(kFull, v < 0);
}

__device__ __forceinline__ uint32_t hash_planes(const uint32_t k[5])
{
    uint32_t h = k[0] * 0x9E3779B1u;
    h ^= k[1] * 0x85EBCA77u;
    h ^= k[2] * 0xC2B2AE3Du;
    h ^= k[3] * 0x27D4EB2Fu;
    h ^= k[4] * 0x165667B1u;
    return h ^ (h >> 15);
}

// ------------------------------------------------------------------------------------
// the mover's view of a lane-distributed position
// ------------------------------------------------------------------------------------
struct Mover {
    int lane, player;
    int unit;             // what one checker of the mover adds to this lane: +-1 on points, +1 on bar/off lanes

    __device__ __forceinline__ Mover(int ln, int pl) : lane(ln), player(pl) { unit = ln < 24 ? (pl ? -1 : 1) : 1; }

    // legal origins of the mover on state v for one die (bgx_core.h legal_origins) from two ballots, in code space
    __device__ __forceinline__ uint32_t legal_here(int v, int die) const
    {
        const int rel = lane < 24 ? v * unit : v;                         // mover-relative count; bar/off lanes as they are
        const uint32_t own = __ballot_sync(kFull, rel > 0);
        const uint32_t blk = __ballot_sync(kFull, rel < -1) & 0xFFFFFFu;  // points the mover cannot land on
        const uint32_t occ = (own & 0xFFFFFFu) << 1, wall = blk << 1;
        const bool on_bar = (own >> (24 + player)) & 1u;
        if (player == 0) {
            if (on_bar) return ((wall >> die) & 1u) ? 0u : 1u;
            uint32_t legal = occ & ((~wall & kPoints) >> die);
            if (occ != 0 && (occ & kP1Outside) == 0) {
                legal |= occ & (1u << (25 - die));
                const int hi = highest_bit(occ);
                if (hi + die > 25) legal |= 1u << hi;
            }
            return legal;
        }
        if (on_bar) return ((wall >> (25 - die)) & 1u) ? 0u : (1u << 25);
        uint32_t legal = occ & ((~wall & kPoints) << die) & kPoints;
        if (occ != 0 && (occ & kP2Outside) == 0) {
            legal |= occ & (1u << die);
            const uint32_t any = (__ballot_sync(kFull, v != 0) & 0xFFFFFFu) << 1;   // either colour (SURVEY A.3 Q4)
            const int hi = highest_bit(any & kP2Window);
            if (hi < die && ((occ >> hi) & 1u)) legal |= 1u << hi;
        }
        return legal;
    }

    // lanes of the origin / destination codes
    __device__ __forceinline__ int src_lane(int o) const { return (o == (player ? 25 : 0)) ? 24 + player : o - 1; }
    __device__ __forceinline__ int dst_lane(int d) const { return (d == (player ? 0 : 25)) ? 26 + player : d - 1; }
    __device__ __forceinline__ int unit_of_points() const { return player ? -1 : 1; }

    // the child state (game.cpp:624-659); dval = what stood on the landing lane
    __device__ __forceinline__ int apply(int v, int o, int d, int &dval) const
    {
        const int src = src_lane(o), dst = dst_lane(d);
        dval = __shfl_sync(kFull, v, dst);
        const bool hit = dst < 24 && dval * unit_of_points() == -1;
        int t = lane == dst ? (hit ? 2 * unit : unit) : 0;
        t -= lane == src ? unit : 0;
        t += (hit && lane == 25 - player) ? 1 : 0;
        return v + t;
    }
};

// ------------------------------------------------------------------------------------
// the turn tree: legalTurnSequences (cppsrc/game.cpp:134-191) + collectDoubles (109-131)
// ------------------------------------------------------------------------------------
// Leaf is called as leaf(state_of_this_lane, packed_moves_with_length, length) once per
// legal turn sequence, in the reference's order, duplicates included.  All control flow
// is warp-uniform; the recursion is a template over the depth and fully inlined, so the
// per-depth state lives in registers.
template <class Leaf>
struct TurnWalk : Mover {
    Leaf &leaf;
    int dieA, dieB;       // die of even / odd depths

    __device__ __forceinline__ TurnWalk(Leaf &lf, int ln, int pl) : Mover(ln, pl), leaf(lf) {}

    template <int D, bool kDbl>
    __device__ __forceinline__ void visit(int v, uint64_t moves)
    {
        constexpr int kMax = kDbl ? 4 : 2;
        uint32_t legal = 0;
        if constexpr (D < kMax) legal = legal_here(v, (D & 1) ? dieB : dieA);
        if (legal == 0) {
            // a node without a move ends the sequence (game.cpp:117-121, 148-151); the root of a
            // non-double pass emits nothing (SURVEY A.3 Q5)
            if (kDbl || D > 0) leaf(v, moves | ((uint64_t)D << 40), D);
            return;
        }
        if constexpr (D < kMax) {
            const int die = (D & 1) ? dieB : dieA;
            do {
                const int o = lowest_bit(legal);
                legal &= legal - 1;
                const int d = destination(player, o, die);
                int dv;
                const int child = apply(v, o, d, dv);
                visit<D + 1, kDbl>(child, moves | pack_move(o, d, D));
            } while (legal);
        }
    }
};

template <class Leaf>
__device__ __forceinline__ void walk_turn(int root, int lane, int player, int d1, int d2, Leaf &leaf)
{
    TurnWalk<Leaf> w(leaf, lane, player);
    if (d1 == d2) {
        w.dieA = w.dieB = d1;
        w.template visit<0, true>(root, 0ull);
    } else {
#pragma unroll 1
        for (int pass = 0; pass < 2; pass++) {          // game.cpp:143-188: d1 first, then d2 first
            w.dieA = pass ? d2 : d1;
            w.dieB = pass ? d1 : d2;
            w.template visit<0, false>(root, 0ull);
        }
    }
}

__device__ __forceinline__ float sigmoid_f32(float z) { return 1.0f / (1.0f + expf(-z)); }

__device__ __forceinline__ float off_feature(int k) { return __fdiv_rn((float)k, 15.0f); } // == (float)(k/15.0), k<=15

// ------------------------------------------------------------------------------------
// shared-memory staging of the weight table: one TMA bulk copy per CTA
// ------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// Every thread of the CTA must call this; returns once the table is visible.
__device__ __forceinline__ void stage_table(void *dst_smem, const void *src_gmem, uint64_t *bar, int bytes)
{
    const uint32_t b = smem_u32(bar);
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(b), "r"(1));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(b), "r"(bytes) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(b)
                     : "memory");
    }
    uint32_t done = 0;
    while (!done) {
        asm volatile("{\n\t.reg .pred p;\n\t"
                     "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                     "selp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done)
                     : "r"(b), "r"(0)
                     : "memory");
    }
}

// ------------------------------------------------------------------------------------
// one greedy / epsilon-greedy ply: make_move (model.py:180-222)
// ------------------------------------------------------------------------------------
struct Choice {
    int v;            // this lane's element of the chosen afterstate
    uint64_t moves;   // packed sequence | length << 40
    float value;
    int n_seq;        // sequences enumerated (reference count)
    int n_scored;     // afterstates sent through the network
    int n_visited;    // tree edges walked (moves applied)
    bool any;         // a sequence exists (N > 0)
    bool z_ok;        // the walker's stash holds the hidden pre-activation of v (greedy_ply with a stash; false otherwise)
};

struct CountLeaf {
    int n = 0;
    __device__ __forceinline__ void operator()(int, uint64_t, int) { n++; }
};

struct PickLeaf {
    int target, n = 0, v = 0;
    uint64_t moves = 0;
    __device__ __forceinline__ explicit PickLeaf(int t) : target(t) {}
    __device__ __forceinline__ void operator()(int vv, uint64_t mv, int)
    {
        if (n == target) { v = vv; moves = mv; }
        n++;
    }
};

// opening position (cppsrc/game.cpp:251) for this lane
__device__ __forceinline__ int start_value(int lane)
{
    // 2 0 0 0 0 -5 0 -3 0 0 0 5 -5 0 0 0 3 0 5 0 0 0 0 -2
    switch (lane) {
    case 0: return 2;
    case 5: return -5;
    case 7: return -3;
    case 11: return 5;
    case 12: return -5;
    case 16: return 3;
    case 18: return 5;
    case 23: return -2;
    default: return 0;
    }
}

// first mover of game `gid`: play_game's roll-off by dice sums (train.py:89-97) on Philox
// stream 1, or the parity rule of benchmark.py:74
__device__ __forceinline__ int first_mover_of(uint32_t k0, uint32_t k1, uint64_t gid, int rule)
{
    if (rule == 1) return (int)(gid & 1);
    for (uint32_t attempt = 0;; attempt++) {
        const Philox r = philox4x32_10(k0, k1, attempt, (uint32_t)gid, (uint32_t)(gid >> 32), 1u);
        const int s1 = die_of(r.x[0]) + die_of(r.x[1]);
        const int s2 = die_of(r.x[2]) + die_of(r.x[3]);
        if (s1 != s2) return s1 > s2 ? 0 : 1;
    }
}

} // namespace bgx
