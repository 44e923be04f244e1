// bgx_ply.cuh — the greedy ply of the fused self-play path.
//
// Contract: make_move (model.py:180-222) — enumerate the legal turn sequences in reference
// order, score every distinct afterstate with the 198-128-1 net, first-index arg-best.
// How the work is done (each step driven by an ncu capture, see profiles/):
//
//  1. DELTA EVALUATION IN FIXED POINT.  The hidden pre-activation z = W1 x + b1 of a node is kept
//     per tree depth; a move changes 2-4 features (one checker leaves a stack, one joins a stack,
//     a hit also flips the blot and the enemy bar), so z(child) = z(parent) +- 2-4 rows of the
//     feature-major weight table: 2-4 LDS.128 + the sigmoid epilogue instead of a walk over all
//     ~16 occupied points.  z is int32 fixed point, which makes it independent of the path (see
//     PlyEvaluator): an afterstate's value is a pure function of the afterstate.
//  2. DEPTH-SPECIALISED WALK IN REGISTERS.  The turn tree is walked by a fully inlined
//     template recursion (one instance per depth), so node state, node z and the origins
//     still to try are registers, not a stack in memory, and work is lazy: a child is only
//     applied and probed in the cache; everything else happens for new afterstates only.
//  3. MEMOISED DOUBLES.  In a double, the same position is reached at the same depth through
//     many move orders (start 3-3: 536 sequences, 73 distinct afterstates).  Interior nodes
//     at depth >= 2 are remembered with the number of sequences below them; meeting one again
//     adds that count to N and skips the whole sub-tree: all its afterstates were already
//     scored earlier in reference order, so the first-index arg-best is unchanged and N stays
//     exact.  The memo shares the per-warp two-way cache with the scored-afterstate set; it is
//     lossy in the safe direction only (a miss re-walks, never mis-counts).
//  4. BYTE-PER-LANE CACHE.  An entry is the position itself, lane l owning byte l; the set
//     index is one REDUX.SUM.  A probe is one byte load per way, one compare, one vote.
//  5. NOTHING PER LANE IS A BRANCH, NOTHING PER WARP IS UNPROVEN.  Selects on the lane are written so that they
//     compile to one LOP3 / SEL (a `lane == 28 ? a : b` inside a template-free helper became BSSY / BRA / BSYNC),
//     and every value the walk branches on is provably warp-uniform for ptxas (ballots, REDUX, shuffles from a fixed
//     lane): otherwise each *_sync intrinsic of the walk is guarded by BRA.DIV (DESIGN 2.1-11; the kernels reconverge
//     before every back-edge for the same reason).
//  6. A MOVE IS (origin lane, landing lane, blot bit).  Origins are lanes throughout the walk (legal masks, twins, the path);
//     they become the reference's origin codes only when the chosen sequence is packed (finish_choice).  A node's moves are
//     computed once for all origins; a child is then one shuffle, two lane tests and a few multiply-adds.
//  7. THE MOVER'S FRAME.  A ply converts its root once so that the mover's checkers are positive and its bar / borne-off lanes are
//     24 / 26 whoever moves (mover_frame), and converts the chosen afterstate back once: a move adds and removes plain ones.
#pragma once
#include <climits>

#include "bgx_device.cuh"

namespace bgx {

constexpr int kPlyEntryBytes = 32;       // one byte per lane: 28 state bytes, node tag, ply generation, sub-tree count, spare

// Per-warp scratch in shared memory: the ply cache, kSets two-way sets of 32-byte entries.  Lane l
// owns byte l of both ways of every set: it alone reads and writes that byte, so the walk needs
// no __syncwarp.
template <int kSets>
struct __align__(16) PlyScratch {
    uint8_t cache[kSets * 2 * kPlyEntryBytes];
};

// 1 / (1 + 2^(-z log2 e)) on the SFU: ex2.approx + rcp.approx (flush-to-zero: 2^x underflows to 0 exactly
// where 1 + 2^x rounds to 1 anyway), ~3e-7 relative error, 4 instructions
__device__ __forceinline__ float fast_sigmoid(float z)
{
    float e, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(z * -1.4426950408889634f));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.0f + e));
    return r;
}

// the same with the 2^x argument already formed: 1 / (1 + 2^a)
__device__ __forceinline__ float sigmoid_exp2(float a)
{
    float e, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(a));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.0f + e));
    return r;
}

// off/15.0 for off = 0..16 (model.py:143-144: float64 divide, stored as float32); [16] pads the k+1 read
__device__ __constant__ float kOffFeature[17] = {
    (float)(0 / 15.0), (float)(1 / 15.0), (float)(2 / 15.0), (float)(3 / 15.0), (float)(4 / 15.0), (float)(5 / 15.0),
    (float)(6 / 15.0), (float)(7 / 15.0), (float)(8 / 15.0), (float)(9 / 15.0), (float)(10 / 15.0), (float)(11 / 15.0),
    (float)(12 / 15.0), (float)(13 / 15.0), (float)(14 / 15.0), (float)(15 / 15.0), (float)(16 / 15.0)};

// ---- the evaluator of the ply kernels: hidden pre-activations in FIXED POINT ---------------
// z = b1 + W1 x is accumulated in int32 with a per-network power-of-two scale S (k_fixed_scale:
// the largest S with |z| S < 2^30 for every reachable position).  Integer addition is associative,
// so the z of a position is the same whichever path of the turn tree led to it, whichever warp
// walked it and whatever the caches held: the value of an afterstate is a pure function of the
// afterstate, duplicates score bit-identically, and the strict first-index arg-best is reproducible
// bit for bit.  (Float accumulation along the tree path differed in the last bits from path to
// path, which made near-ties between distinct afterstates depend on timing.)  Resolution: 2^-30
// of the largest possible |z|, finer than fp32's own rounding of a sum of that size.
// Table Ti[198][128] (k_build_fixed), per feature row f:
//   unit features (f < 192, f % 4 != 3), turn flags 192/193     round(W1[:,f] S)
//   slope features (f % 4 == 3): (n-3)/2 grows by 1/2 per checker   round(W1[:,f] S / 2), coefficient +-1
//   bar features 194/195: n/2                                       round(W1[:,f] S / 2), coefficient +-1
//   borne-off features 196/197: k/15 is not a multiple of a step    the fp32 weight itself (bit pattern);
//                                                                   contribution T(k) = round(W1 (fl(k/15) S)), a function of k
//   rows 198 + 15 p + k (k = 0..14): T(k+1) - T(k) of player p      what the (k+1)-th borne-off checker adds
//   row 228: round(b1 S); row 229: w2; row 230: {S, 1/S, b2, 0} in every lane
//                                                    the evaluator's constants are read where needed instead of living in registers
struct PlyEvaluator {
    const int4 *T4;      // shared memory, fixed-point table Ti[231][32] int4

    __device__ __forceinline__ static void add(int4 &z, const int4 &t) { z.x += t.x; z.y += t.y; z.z += t.z; z.w += t.w; }
    __device__ __forceinline__ static void sub(int4 &z, const int4 &t) { z.x -= t.x; z.y -= t.y; z.z -= t.z; z.w -= t.w; }
    __device__ __forceinline__ static void addn(int4 &z, int n, const int4 &t) { z.x += n * t.x; z.y += n * t.y; z.z += n * t.z; z.w += n * t.w; }
    // contribution of k borne-off checkers of `player` (row 196 + player holds the fp32 weights)
    __device__ __forceinline__ int4 off_term(int k, int player, int lane) const
    {
        const int4 w = T4[(196 + player) * 32 + lane];
        const float f = kOffFeature[k] * __int_as_float(T4[kRowConst * 32 + lane].x);   // same expression as k_build_fixed
        return make_int4(__float2int_rn(__int_as_float(w.x) * f), __float2int_rn(__int_as_float(w.y) * f),
                         __float2int_rn(__int_as_float(w.z) * f), __float2int_rn(__int_as_float(w.w) * f));
    }
    // pre-activation of a position from scratch (the root of a ply; k_evaluate)
    __device__ __forceinline__ int4 preactivation(int v, int lane, int turn) const
    {
        const int n = v < 0 ? -v : v;
        const int packed = (8 * lane + (v > 0 ? 0 : 4)) | (n << 8);
        uint32_t occ = __ballot_sync(kFull, lane < 24 && v != 0);
        int4 z = T4[kRowB1 * 32 + lane];
        while (occ) {
            const int i = lowest_bit(occ);
            occ &= occ - 1;
            const int p = __shfl_sync(kFull, packed, i);
            const int base = p & 0xFF, cnt = p >> 8;
            const int4 *row = T4 + base * 32 + lane;
            add(z, row[0]);
            if (cnt >= 2) add(z, row[32]);
            if (cnt >= 3) add(z, row[64]);
            if (cnt >= 4) addn(z, cnt - 3, row[96]);
        }
        add(z, T4[(192 + turn) * 32 + lane]);
        const int bar1 = __shfl_sync(kFull, v, 24), bar2 = __shfl_sync(kFull, v, 25);
        const int off1 = __shfl_sync(kFull, v, 26), off2 = __shfl_sync(kFull, v, 27);
        if (bar1) addn(z, bar1, T4[194 * 32 + lane]);
        if (bar2) addn(z, bar2, T4[195 * 32 + lane]);
        if (off1) add(z, off_term(off1, 0, lane));
        if (off2) add(z, off_term(off2, 1, lane));
        return z;
    }
    // hidden layer -> output.  The sigmoid's 2^x argument is z * (-log2(e) / S) in ONE multiply; the 32 lane sums of w2 . h are
    // added as integers at scale Y (one REDUX.SUM instead of five shuffle + add rounds; order-independent, so V stays a pure
    // function of the position).  Resolution 2^-30 of sum |w2|: ~1e-7 of V in the worst case.
    // output_sum: the integer the value is a function of; value_of: V.  V is a NON-DECREASING function of the sum (an FFMA, a
    // multiply, ex2.approx, an add, rcp.approx: each monotone - for the two SFU approximations that is checked exhaustively on
    // the device, bgx_sfu_monotone / test_sfu_approximations_are_monotone), so the walk compares sums and evaluates V only for
    // a sum that beats the best one so far: the strict first-index arg-best over V is unchanged.
    __device__ __forceinline__ int output_sum(const int4 &zi, int lane) const
    {
        const int4 wi = T4[kRowW2 * 32 + lane], ci = T4[kRowConst * 32];       // (one address for the warp: the value is provably uniform)
        const float c = __int_as_float(ci.y), Y = __int_as_float(ci.w);
        const float y = __int_as_float(wi.x) * sigmoid_exp2((float)zi.x * c) + __int_as_float(wi.y) * sigmoid_exp2((float)zi.y * c) +
                        __int_as_float(wi.z) * sigmoid_exp2((float)zi.z * c) + __int_as_float(wi.w) * sigmoid_exp2((float)zi.w * c);
        return __reduce_add_sync(kFull, __float2int_rn(y * Y));
    }
    __device__ __forceinline__ float value_of(int total) const
    {
        const int4 ci = T4[kRowConst * 32];
        const float inv_y = __int_as_float(0x7F000000 - ci.w);                    // Y is a power of two
        return fast_sigmoid(fmaf((float)total, inv_y, __int_as_float(ci.z)));
    }
    __device__ __forceinline__ float finish(const int4 &zi, int lane) const { return value_of(output_sum(zi, lane)); }
};

// a row of the table by its 32-bit shared-memory address (the walk's addresses are formed as plain integers: no generic-pointer
// window arithmetic per row).  volatile: otherwise the loop-invariant rows of a hit are hoisted out of the walk's loops and held
// in registers (k_select<20,86> then spills)
__device__ __forceinline__ int4 lds128(uint32_t a)
{
    int4 r;
    asm volatile("ld.shared.v4.s32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(a));
    return r;
}

// The per-warp cache of one ply.  Two kinds of entries share it:
//   tag 0      an afterstate that was already scored in this ply (the exact-duplicate filter)
//   tag 2, 3   an interior node of a double at that depth, with the number of sequences below it
// An entry is the position itself, one byte per lane, so a probe is one byte load per way, one
// compare and one vote; the set index comes from a single warp-wide integer reduction
// (REDUX.SUM) of value x per-lane multiplier.  A hit is an exact match of all 28 state bytes,
// the tag and the ply generation, so the cache can only lose time, never exactness.
template <int kSets>
struct PlyCache {
    uint8_t *col;        // this lane's byte column of the cache (slots + lane)
    uint32_t meta;       // this lane's byte of a tag-0 entry above the state bytes: lane 29 the ply generation (1..255, bumped per
                         // ply; stale entries are the preferred victims), every other lane 0 (lanes 28..31 of a position hold 0)
    const uint32_t *kmul;// this lane's hash multiplier, in the evaluator's table (row kRowLane): one LDS per probe - held in a
                         // register the compiler recomputed it from the lane at every probe (5 ALU instructions, 3 % of the kernel)

    struct Probe {
        uint32_t off;    // byte offset of the set
        uint32_t m0, m1; // per-lane equality masks of way 0 / way 1
        uint32_t h, got0, got1;
        __device__ __forceinline__ bool hit() const { return m0 == kFull || m1 == kFull; }
    };

    __device__ __forceinline__ void clear(int lane) const
    {
        uint32_t *w = reinterpret_cast<uint32_t *>(col - lane);
        for (int i = lane; i < kSets * 2 * kPlyEntryBytes / 4; i += 32) w[i] = 0;
    }
    __device__ __forceinline__ void reset(uint8_t *p, const int4 *T4, int lane)
    {
        col = p + lane;
        meta = 0;
        kmul = reinterpret_cast<const uint32_t *>(T4 + kRowLane * 32) + lane;
        clear(lane);
    }
    __device__ __forceinline__ void next_ply(int lane)
    {
        uint32_t gen = (__shfl_sync(kFull, meta, 29) + 1) & 0xFFu;
        if (gen == 0) {
            clear(lane);
            gen = 1;
            __syncwarp();
        }
        meta = lane == 29 ? gen : 0u;
    }
    // what this lane's byte of a matching entry holds: a state byte, the node tag (lane 28), the generation (lane 29), the
    // sub-tree count of a memo entry (lane 30, not compared), 0 (lane 31)
    template <int kTag>
    __device__ __forceinline__ uint32_t byte_of(int v, int lane) const
    {
        uint32_t b = ((uint32_t)v & 0xFFu) | meta;
        if (kTag != 0) b |= lane == 28 ? (uint32_t)kTag : 0u;
        return b;
    }
    template <int kTag>
    __device__ __forceinline__ Probe probe(int v, int lane) const
    {
        Probe p;
        // the high bits of a sum of products are its best-mixed ones: they pick the set, bit 20 the random victim
        const uint32_t h = __reduce_add_sync(kFull, (uint32_t)v * *kmul) + (uint32_t)kTag * 0x9E3779B1u;
        p.h = h;
        p.off = __umulhi(h, (uint32_t)kSets) * (2 * kPlyEntryBytes);
        const uint8_t *e = col + p.off;
        p.got0 = e[0];
        p.got1 = e[kPlyEntryBytes];
        const uint32_t mine = byte_of<kTag>(v, lane);
        p.m0 = __ballot_sync(kFull, p.got0 == mine);
        p.m1 = __ballot_sync(kFull, p.got1 == mine);
        if (kTag != 0) { p.m0 |= 0x40000000u; p.m1 |= 0x40000000u; }       // a memo entry's count is not part of the key
        return p;
    }
    // after a miss.  Victim: a way left over from an earlier ply (bit 29 of its mask: the generation differs), else pseudo-random
    template <int kTag>
    __device__ __forceinline__ void write(const Probe &p, int v, int count, int lane) const
    {
        const uint32_t way = (p.m0 >> 29) & (~(p.m1 >> 29) | (p.h >> 20)) & 1u;
        uint32_t mine = byte_of<kTag>(v, lane);
        if (kTag != 0) mine |= lane == 30 ? (uint32_t)count : 0u;
        col[p.off + way * kPlyEntryBytes] = (uint8_t)mine;
    }
    // memo of interior nodes (tag = depth): sub-tree sequence count (<= 225), or -1
    template <int kTag>
    __device__ __forceinline__ int lookup(int v, int lane) const
    {
        const Probe p = probe<kTag>(v, lane);
        const int cnt = (int)__shfl_sync(kFull, p.m0 == kFull ? p.got0 : p.got1, 30);
        return p.hit() ? cnt : -1;
    }
    // (the node cannot be in the cache: its lookup missed, and the walk below it stored deeper tags only)
    template <int kTag>
    __device__ __forceinline__ void store(int v, int count, int lane) const
    {
        if (count > 255) return;                      // cannot happen (<= 15 x 15 sequences below depth 2); never mis-count
        const Probe p = probe<kTag>(v, lane);
        if (!p.hit()) write<kTag>(p, v, count, lane);
    }
};

// The greedy walk sees every position in the MOVER'S FRAME (DESIGN 2.1-20): for PLAYER2 the point lanes are negated and the
// bar lanes (24, 25) and borne-off lanes (26, 27) swap, so the mover's checkers are positive, its bar is lane 24 and its
// borne-off count lane 26 whoever moves.  Points keep their lanes (ascending lanes stay the reference's origin order for both
// players); the direction of travel and the bear-off rules stay per player.  The map is its own inverse.
__device__ __forceinline__ int mover_frame(int v, int lane, int player)
{
    const int w = __shfl_sync(kFull, v, player && (unsigned)(lane - 24) < 4u ? lane ^ 1 : lane);
    return player && lane < 24 ? -w : w;
}

// A sequence that ends before the dice are used up (no legal move left) is the rare kind of leaf.  Its
// afterstate is scored FROM SCRATCH by this out-of-line routine - the fixed-point z of a position does not
// depend on how it is computed - so the fully inlined walk carries the leaf code only at its last level
// (the kernel's code has to stay close to the 32 KB instruction cache).  v is in the mover's frame.  Returns the output sum,
// kSeenBefore if scored before.
constexpr int kSeenBefore = INT_MIN;
template <int kSets>
__device__ __noinline__ int score_early_leaf(uint8_t *col, uint32_t meta, const uint32_t *kmul, const int4 *T4, int v, int lane, int player)
{
    PlyCache<kSets> cache;
    cache.col = col; cache.meta = meta; cache.kmul = kmul;
    const typename PlyCache<kSets>::Probe pr = cache.template probe<0>(v, lane);
    if (pr.hit()) return kSeenBefore;
    cache.template write<0>(pr, v, 0, lane);
    PlyEvaluator e;
    e.T4 = T4;
    return e.output_sum(e.preactivation(mover_frame(v, lane, player), lane, player), lane);
}

// ---- the walk ----------------------------------------------------------------------------
// One template instance per tree depth (the recursion is fully inlined), so the per-depth
// state of the walk - node state, node pre-activation, origins still to try - lives in
// registers and every level knows at compile time which die it plays and whether its children
// can have children.  Work is done as late as possible: a child is first only APPLIED (one
// shuffle for the landing point, three predicated adds) and probed in the cache; the rows its
// move changes in the network input, its pre-activation and its value are computed only for
// afterstates that were not scored yet in this ply and for interior nodes.
// Every state of the walk is in the mover's frame (mover_frame): the mover's checkers count +1 wherever they stand, so a move
// adds and removes plain ones and the player is left only in the direction of travel, the bear-off rules, the table rows and
// the value's sign, all uniform per ply.
template <int kSets>
struct PlyWalk {
    const PlyEvaluator &ev;
    const PlyCache<kSets> &cache;
    int lane, player;
    uint32_t Tme;         // shared address of this lane's column of the evaluator's table, from the mover's feature block on (child_z)
    int dieA, dieB;       // die of even / odd depths
    uint32_t root_only;   // restricts the root's origin lanes (all ones: no restriction)
    uint32_t twin_root;   // non-doubles, second pass: the root origin lanes of the FIRST pass' first die (0 in the first pass)
    bool nd;              // a pass of a NON-double: walked by the last two levels (2, 3 -> leaves at 4) of the one walk there is,
                          // so that the kernel carries one copy of the per-depth code instead of two (instruction cache)
    int4 zroot;
    int4 *zstash;         // where this lane keeps the pre-activation of the best afterstate so far (nullptr: nowhere), and
    bool z_ok;            // whether it is there: the next ply of the game starts from it instead of summing ~30 rows again
    // result
    float best_key;       // value, negated for PLAYER2 (who minimises): always maximised, strict > keeps the first
    int best_sum;         // the output sum behind it (negated likewise): a sum that does not beat it cannot beat the value
    int best_v;
    uint32_t best_path;   // origin lanes 5 bits each, length << 20
    int n_seq, n_scored, n_visited;

    __device__ __forceinline__ PlyWalk(const PlyEvaluator &e, const PlyCache<kSets> &c, int ln, int pl)
        : ev(e), cache(c), lane(ln), player(pl)
    {
        Tme = smem_u32(e.T4 + ln + (pl ? 4 * 32 : 0));
        root_only = kFull;
        twin_root = 0;
        nd = false;
        best_key = __int_as_float(0xff800000);          // -inf
        best_sum = INT_MIN;
        best_v = 0; best_path = 0;
        n_seq = n_scored = n_visited = 0;
        zstash = nullptr; z_ok = false;
    }

    // What moving one checker does, as a word: bits 0..4 the landing lane | bits 5..12 the row the origin loses | bits 23..30 the
    // row the landing lane gains | bit 31 a hit.  The fields sit where a child reads them with few instructions: the landing lane
    // is XOR-compared with the lane in place, the low 13 bits masked to the origin row are that row's offset / 16, the hit is the
    // sign.  Rows are rows of Tme = this lane's column of the table shifted to the MOVER's feature block (row
    // 8 p + k of Tme: "k + 1 checkers of the mover on point p"; the other rows follow from the player by one multiply-add).
    // src / dst: the origin and landing lanes (bar 24, borne off 26), sval / dval: what stands there.
    __device__ __forceinline__ uint32_t move_word(int sval, int dval, int src, int dst) const
    {
        const int row_src = src >= 24 ? 194 - 3 * player : 8 * src + (sval < 4 ? sval : 4) - 1;      // (194 + player) - 4 player
        const bool hit = dval == -1;                                     // (only points hold the enemy's checkers, negative)
        int row_dst = dst >= 24 ? kFeatures + 11 * player + dval : 8 * dst + (dval < 3 ? dval : 3);  // (198 + 15 player) - 4 player
        if (hit) row_dst = 8 * dst;
        return (uint32_t)dst | ((uint32_t)row_src & 0xFFu) << 5 | ((uint32_t)row_dst & 0xFFu) << 23 | (hit ? 1u << 31 : 0u);
    }
    // ... for ALL origins of a node at once: lane l computes the word of "the checker on lane l moves by the node's die" (a garbage
    // word where no legal origin stands); a child then costs one shuffle instead of this arithmetic per child
    __device__ __forceinline__ uint32_t node_moves(int v, int die) const
    {
        const int d = lane + die * dir();                                // from a point: the landing point, or off the board
        int dl = (unsigned)d > 23u ? 26 : d;
        if (lane >= 24) dl = player ? 24 - die : die - 1;                // from the bar (game.cpp:89-97)
        return move_word(v, __shfl_sync(kFull, v, dl), lane, dl);
    }
    // the child state (game.cpp:624-659): the checker leaves lane sl and lands where the word says
    __device__ __forceinline__ int apply_word(int v, int sl, uint32_t mv) const
    {
        const int hit = (int)(mv >> 31);
        int t = v + (lane == 25 ? hit : 0);                                  // a hit sends the blot to the enemy's bar ...
        t += ((mv ^ (uint32_t)lane) & 31u) == 0u ? 1 + hit : 0;              // ... where the checker lands
        t -= lane == sl ? 1 : 0;
        return t;
    }
    __device__ __forceinline__ int dir() const { return player ? -1 : 1; }   // direction of travel on the point lanes

    // legal origin lanes of the mover for one die (bgx_core.h legal_origins in the mover's frame): bit l = the checker on lane l
    // may move, the bar is lane 24.  Points keep their order (lane = code - 1), and a mover on the bar has the bar as its only
    // origin, so ascending lanes are the reference's order.
    __device__ __forceinline__ uint32_t legal_lanes(int v, int die) const
    {
        const uint32_t own = __ballot_sync(kFull, v > 0);
        const uint32_t wall = __ballot_sync(kFull, v < -1) & 0xFFFFFFu;    // points the mover cannot land on
        const uint32_t occ = own & 0xFFFFFFu;
        if ((own >> 24) & 1u) return ((wall >> (player ? 24 - die : die - 1)) & 1u) ? 0u : 1u << 24;
        if (player == 0) {
            uint32_t legal = occ & ((~wall & 0xFFFFFFu) >> die);
            if (occ != 0 && (occ & (kP1Outside >> 1)) == 0) {
                legal |= occ & (1u << (24 - die));
                const int hi = highest_bit(occ);
                if (hi + die > 24) legal |= 1u << hi;
            }
            return legal;
        }
        uint32_t legal = occ & ((~wall & 0xFFFFFFu) << die);
        if (occ != 0 && (occ & (kP2Outside >> 1)) == 0) {
            legal |= occ & (1u << (die - 1));
            const uint32_t any = __ballot_sync(kFull, v != 0) & 0xFFFFFFu;   // either colour (SURVEY A.3 Q4)
            const int hi = highest_bit(any & (kP2Window >> 1));
            if (hi < die - 1 && ((occ >> hi) & 1u)) legal |= 1u << hi;
        }
        return legal;
    }

    // pre-activation of the child reached from zpar by the move mv: 2 rows, 4 after a hit (a row is 512 bytes)
    __device__ __forceinline__ int4 child_z(const int4 &zpar, uint32_t mv) const
    {
        int4 z = zpar;
        PlyEvaluator::sub(z, lds128(Tme + ((mv & 0x1FE0u) << 4)));          // one checker less on the origin (or the bar)
        if ((int)mv < 0) {                                                  // a hit
            const uint32_t dst = mv & 31u;
            PlyEvaluator::sub(z, lds128(Tme + (8 * dst + 4 - 8 * player) * 512));   // the blot leaves (the enemy's block: +4 / -4) ...
            PlyEvaluator::add(z, lds128(Tme + (195 - 5 * player) * 512));           // ... for the enemy's bar: (195 - player) - 4 player
        }
        PlyEvaluator::add(z, lds128(Tme + ((mv >> 14) & 0x1FE00u)));         // one more on the landing point (or borne off)
        return z;
    }

    // a legal turn sequence ends on v (reference order); score it unless this exact state was scored before
    template <int D>
    __device__ __forceinline__ void leaf(int v, const int4 &zpar, uint32_t mv, uint32_t path)
    {
        n_seq++;
        const typename PlyCache<kSets>::Probe pr = cache.template probe<0>(v, lane);
        if (pr.hit()) return;
        cache.template write<0>(pr, v, 0, lane);
        const int4 z = D == 0 ? zroot : child_z(zpar, mv);
        const int total = ev.output_sum(z, lane);
        n_scored++;
        const int sum = player ? -total : total;
        if (sum > best_sum) {
            const float val = ev.value_of(total);
            const float key = player ? -val : val;
            if (key > best_key) {
                best_key = key; best_sum = sum; best_v = v; best_path = path | ((uint32_t)D << 20);
                if (zstash) { *zstash = z; z_ok = true; }
            }
        }
    }

    __device__ __forceinline__ void early_leaf(int v, uint32_t path_and_len)
    {
        n_seq++;
        // (a call's result counts as divergent: the shuffle makes the branches below uniform ones, see k_selfplay)
        const int total = __shfl_sync(kFull, score_early_leaf<kSets>(cache.col, cache.meta, cache.kmul, ev.T4, v, lane, player), 0);
        if (total == kSeenBefore) return;
        n_scored++;
        const int sum = player ? -total : total;
        if (sum > best_sum) {
            const float val = ev.value_of(total);
            const float key = player ? -val : val;
            if (key > best_key) { best_key = key; best_sum = sum; best_v = v; best_path = path_and_len; z_ok = false; }
        }
    }

    // Twins.  Two on-board moves of one turn commute: played in either order they remove the same two checkers, land on the
    // same two points and hit the same blots (walls do not change during a turn, only bar entry and bearing off depend on the
    // rest of the board).  So under a node reached by the on-board move o, the last move o' leads to the position that
    // (.., o', o) leads to whenever o' was already playable BEFORE o: in a double when o' is a smaller origin of the parent
    // node, in the second pass of a non-double when o' is a root origin of the first pass.  The reference visits that twin
    // EARLIER (ascending origins; first pass first), it has the same value, and the strict first-index arg-best can never
    // prefer the later copy: such leaves are counted, not walked.  `legal_par` = all origins of the parent node.  (In lane space
    // "smaller" is "a lower lane": the orders differ only at the bar, and a mover on the bar has no other origin.)
    // (v, path) = the node; zpar its parent's pre-activation, mv the word of the move that led here (path holds its origin lane),
    // left: that move bore a checker off (kept apart from mv: it steers the walk and has to be provably warp-uniform)
    template <int D>
    __device__ __forceinline__ void visit(int v, const int4 &zpar, uint32_t mv, bool left, uint32_t path, uint32_t legal_par = 0)
    {
        constexpr int kMax = 4;
        uint32_t legal = 0;
        if constexpr (D < kMax) {
            if (D == 1 && nd) legal = 1u;                    // a non-double pass enters at level 2: level 1 hands the root through
            else legal = legal_lanes(v, (D & 1) ? dieB : dieA);
            if (D == 0) legal &= root_only;
        }
        uint32_t twins = 0;
        if constexpr (D == kMax - 1) {
            const int die = (D & 1) ? dieB : dieA;
            const int o = (int)((path >> (5 * (D - 1))) & 31u);
            twins = legal & (nd ? twin_root : legal_par & ((1u << o) - 1u));
            twins &= player ? ~((1u << die) - 1u) : ((1u << (24 - die)) - 1u) | (1u << 24);   // the last move stays on the board ...
            if (left) twins = 0;                                                 // ... and so did the one before it
        }
        if (legal == 0) {
            // a node without a move ends the sequence (game.cpp:117-121, 148-151); the root of a
            // non-double pass emits nothing (SURVEY A.3 Q5)
            if constexpr (D == kMax) leaf<D>(v, zpar, mv, path);
            else if (!(D == 2 && nd)) early_leaf(v, path | ((uint32_t)D << 20));
            return;
        }
        if constexpr (D < kMax) {
            if constexpr (D >= 2) {                          // doubles: same position, same dice left: seen before?
                if (!nd) {
                    const int below = cache.template lookup<D>(v, lane);
                    if (below >= 0) { n_seq += below; return; }
                }
            }
            const int entered = n_seq;
            const uint32_t legal_all = legal;
            n_seq += __popc(twins);                          // counted, not walked (the count below stays path-independent)
            legal &= ~twins;
            if (D == kMax - 1 && legal == 0) {               // every sequence below is an earlier one's twin
                if constexpr (D >= 2) { if (!nd) cache.template store<D>(v, n_seq - entered, lane); }
                return;
            }
            int4 z = zroot;                                  // the root of the turn: of a double at depth 0, of a non-double pass at 2
            if (D != 0 && !(D <= 2 && nd)) z = child_z(zpar, mv);
            const int die = (D & 1) ? dieB : dieA;
            const uint32_t moves = (D == 1 && nd) ? 0u : node_moves(v, die);
            if (!(D == 1 && nd)) n_visited += __popc(legal);      // the moves applied below
            do {
                const int sc = lowest_bit(legal);
                legal &= legal - 1;
                int child = v;
                uint32_t mc = 0;
                bool off = false;
                if (!(D == 1 && nd)) {
                    mc = __shfl_sync(kFull, moves, sc);
                    child = apply_word(v, sc, mc);
                    if (D + 1 == kMax - 1) off = sc < 24 && (unsigned)(sc + die * dir()) > 23u;  // (game.cpp:89-97)
                }
                visit<D + 1>(child, z, mc, off, path | ((uint32_t)sc << (5 * D)), legal_all);
            } while (legal);
            if constexpr (D >= 2) { if (!nd) cache.template store<D>(v, n_seq - entered, lane); }
        }
    }
};

// ---- sharing the sub-trees of a big double inside the CTA --------------------------------
// A double with many first moves has a turn tree of up to ~12 k sequences: walked by one warp
// it is the tail of every launch.  The owner of such a ply PUBLISHES the origins of its root in
// its shared-memory slot and pops them lowest first; warps of the same CTA that have run out of
// queue work pop the highest one, walk that sub-tree with their own cache and deliver the result;
// the owner merges.  Exactness: every root child is walked by exactly one warp in reference
// order, the merge prefers the better value and, on equal values, the lower root origin, which
// is the reference's first-index rule (model.py:212-213); N is the sum of the parts.
constexpr int kStealMinChildren = 4;     // root origins from which a double is worth publishing
constexpr int kGiantMinChildren = 10;    // ... and from which its CTA helps at once wherever the double sits in the queue
// (ShareCtx::urgent_min / urgent_from: the same for smaller doubles from a queue position on - a one-ply launch wants
// that everywhere, a many-ply launch only in its last stretch, because helpers re-score what the owner's cache holds)
constexpr int kStealMaxResults = 16;     // >= the 15 origins a root can have

struct StealSlot {                       // shared memory, one per warp
    uint32_t legal0;                     // root origins nobody has taken yet (0: nothing to take)
    int32_t pending;                     // taken sub-trees still being walked by helpers
    uint32_t nres;                       // results delivered for the current ply
    uint32_t meta;                       // player | die << 8
    int8_t root[32];
};

struct __align__(16) StealResult {       // global memory, [CTA][warp][kStealMaxResults]
    float value;
    int32_t any, n_seq, n_scored, n_visited, origin;
    unsigned long long moves;
    int8_t v[32];
};

template <int kWarps>
struct StealShared {
    StealSlot slot[kWarps];
    int32_t active;                      // warps that still own queue work
    uint32_t urgent;                     // warps whose published double is so big that the others help before claiming new work
    int32_t pad[2];
    unsigned long long stats[8];         // the CTA's share of the launch statistics (kept out of the warps' registers)
};

// what a warp needs to publish its doubles: its slot, its result area, the CTA's urgent mask and its bit in it
struct ShareCtx {
    StealSlot *slot;
    StealResult *results;
    uint32_t *urgent;
    uint32_t my_bit;
    const unsigned long long *queue;     // the launch's work-queue counter ...
    unsigned long long urgent_from;      // ... and the position from which big doubles are urgent
    int urgent_min;                      // root origins that make a double "big" for that purpose
    int giant_min;                       // root origins from which a double is urgent wherever it sits in the queue
};

// best_path holds origin LANES; the packed moves carry the reference's origin codes (the bar: 0 for PLAYER1, 25 for PLAYER2)
__device__ __forceinline__ Choice finish_choice(const uint32_t best_path, float best_key, int best_v, int n_seq, int n_scored,
                                                int n_visited, int root, int player, int d1, int d2, uint32_t best_pass)
{
    Choice best;
    best.any = n_seq > 0;
    best.v = best.any ? best_v : root;
    best.value = best.any ? (player ? -best_key : best_key) : __int_as_float(0x7fc00000);
    best.n_seq = n_seq; best.n_scored = n_scored; best.n_visited = n_visited;
    uint64_t mv = 0;
    if (best.any) {
        const int len = (int)(best_path >> 20);
        mv = (uint64_t)len << 40;
        for (int j = 0; j < len; j++) {
            const int l = (int)((best_path >> (5 * j)) & 31u);
            const int o = l >= 24 ? 25 * player : l + 1;
            const int die = ((j & 1) != (int)best_pass) ? d2 : d1;
            mv |= pack_move(o, destination(player, o, die), j);
        }
    }
    best.moves = mv;
    best.z_ok = false;
    return best;
}

// root_only: bit mask over the root's origin lanes (a helper walks one stolen child); kFull = the whole turn.
// slot/results: the caller's sharing slot (nullptr: never publish).
// zstash: this lane's 16 bytes for the pre-activation of the best afterstate (nullptr: none); carry: it holds the
// pre-activation of `root` as the PREVIOUS mover's walk scored it (same game, one ply earlier): fixed-point sums do not depend
// on how they were formed, so flipping the turn flag gives exactly what preactivation() would compute.
// root and the returned Choice are in the real frame; the walk runs in the mover's (mover_frame: one conversion each way per
// ply).  A published double's root stays in the real frame: a helper's greedy_ply converts it and delivers in the real frame.
template <int kSets>
__device__ __forceinline__ Choice greedy_ply(int root, int lane, int player, int d1, int d2, const PlyEvaluator &ev,
                                             PlyCache<kSets> &cache, uint32_t root_only = kFull, const ShareCtx *share = nullptr,
                                             int4 *zstash = nullptr, bool carry = false)
{
    StealSlot *slot = share ? share->slot : nullptr;
    StealResult *results = share ? share->results : nullptr;
    cache.next_ply(lane);
    PlyCache<kSets> fcache = cache;
    if (player) fcache.kmul += 32;                                       // the hash multipliers of PLAYER2's frame (kRowLane)
    const int froot = mover_frame(root, lane, player);
    PlyWalk<kSets> w(ev, fcache, lane, player);
    w.root_only = root_only;
    if (carry) {
        int4 z = *zstash;
        PlyEvaluator::sub(z, ev.T4[(193 - player) * 32 + lane]);         // the turn flag of the ply before ...
        PlyEvaluator::add(z, ev.T4[(192 + player) * 32 + lane]);         // ... and of this one (model.py:139-140)
        w.zroot = z;
    } else {
        w.zroot = ev.preactivation(root, lane, player);
    }
    w.zstash = zstash;
    uint32_t best_pass = 0;
    bool shared = false;
    // One loop, ONE call site of the walk (every call site would be another inlined copy of all its levels): a double
    // iterates over its root origins (its own, or the ones its helpers leave it), a non-double over its two passes.
    const bool dbl = d1 == d2;
    uint32_t legal = 0;
    float key1 = 0.f;
    int pass = 0;
    w.dieA = d1; w.dieB = d2;
    w.nd = !dbl;
    if (dbl) {
        legal = w.legal_lanes(froot, d1) & root_only;
        if (legal == 0) {
            w.early_leaf(froot, 0u);                                     // no move at all: the empty sequence (SURVEY A.3 Q6)
        } else {
            shared = slot != nullptr && __popc(legal) >= kStealMinChildren;
            if (shared) {                                                // publish the root's origins
                slot->root[lane] = (int8_t)root;
                if (lane == 0) { slot->meta = (uint32_t)player | ((uint32_t)d1 << 8); slot->nres = 0; }
                __threadfence_block();
                __syncwarp();
                if (lane == 0) {
                    atomicExch(&slot->legal0, legal);
                    // near the end of the queue a huge double is the tail of the launch: ask for help at once
                    const int kids = __popc(legal);
                    if (kids >= share->giant_min ||
                        (kids >= share->urgent_min && *(volatile const unsigned long long *)share->queue >= share->urgent_from))
                        atomicOr(share->urgent, share->my_bit);
                }
                __syncwarp();                                            // reconverged before the loop below (see k_selfplay)
            }
        }
    }
    const uint32_t root_moves = dbl ? w.node_moves(froot, d1) : 0u;
    for (;;) {
        int child = froot, oc = 0;
        uint32_t mroot = 0;
        if (dbl) {
            uint32_t bit = 0;
            if (shared) {                                                // pop the lowest origin still there
                // (the whole warp runs the retry loop and every exit is decided by a broadcast value: a loop inside a
                // lane-0 block that an atomic's result ends makes ptxas treat all that follows as diverged, see k_selfplay)
                for (;;) {
                    const uint32_t old = *(volatile uint32_t *)&slot->legal0;
                    if (old == 0) break;
                    const uint32_t low = old & (0u - old);
                    uint32_t was = 0;
                    if (lane == 0) was = atomicAnd(&slot->legal0, ~low);
                    was = __shfl_sync(kFull, was, 0);
                    if (was & low) { bit = low; break; }
                }
            } else {
                bit = legal & (0u - legal);
                legal &= legal - 1;
            }
            if (bit == 0) break;
            oc = lowest_bit(bit);
            mroot = __shfl_sync(kFull, root_moves, oc);
            child = w.apply_word(froot, oc, mroot);
            w.n_visited++;
        } else {                                                         // game.cpp:143-188: d1 first, then d2 first
            if (pass == 2) break;
            w.dieA = pass ? d2 : d1;
            w.dieB = pass ? d1 : d2;
            if (pass) { key1 = w.best_key; w.twin_root = w.legal_lanes(froot, d1); }
            pass++;
        }
        w.template visit<1>(child, w.zroot, mroot, false, (uint32_t)oc);
    }
    if (dbl) {
        if (shared && lane == 0) atomicAnd(share->urgent, ~share->my_bit);
    } else {
        best_pass = w.best_key > key1 ? 1u : 0u;
        // levels 2, 3 wrote the origins at bits 10.. and counted the two levels above into the length
        w.best_path = ((w.best_path & 0xFFFFFu) >> 10) | (((w.best_path >> 20) - 2u) << 20);
    }
    Choice best = finish_choice(w.best_path, w.best_key, mover_frame(w.best_v, lane, player), w.n_seq, w.n_scored, w.n_visited, root, player, d1, d2, best_pass);
    best.z_ok = best.any && w.z_ok;
    if (shared) {
        // wait for the helpers, then merge their sub-trees: better value, then lower root origin
        while (*(volatile int32_t *)&slot->pending != 0) __nanosleep(64);
        __threadfence_block();
        const int n = (int)*(volatile uint32_t *)&slot->nres;
        int best_origin = best.any ? (int)(best.moves & 31u) : 99;
        for (int i = 0; i < n; i++) {
            const StealResult *r = results + i;
            const int any = __ldcg(&r->any);
            best.n_seq += __ldcg(&r->n_seq);
            best.n_scored += __ldcg(&r->n_scored);
            best.n_visited += __ldcg(&r->n_visited);
            if (!any) continue;
            const float val = __ldcg(&r->value);
            const int org = __ldcg(&r->origin);
            const bool better = !best.any || (player ? val < best.value : val > best.value) || (val == best.value && org < best_origin);
            if (better) {
                best.any = true; best.value = val; best_origin = org; best.z_ok = false;
                best.moves = __ldcg(&r->moves);
                best.v = (int)__ldcg(reinterpret_cast<const signed char *>(r->v) + lane);
            }
        }
    }
    return best;
}

// What a warp does once the work queue is empty: help the owners of published doubles in its CTA
// until no warp of the CTA owns queue work any more.  take_child() returns the origin bit it took
// from warp `vw` (filling root / player / die), 0 when there is nothing to take right now, and
// sets `done` once every warp of the CTA has left the queue.
template <int kWarps>
__device__ __forceinline__ uint32_t take_child(StealShared<kWarps> *sh, int lane, int &vw, int &root, int &player, int &die, bool &done,
                                               bool urgent_only = false)
{
    done = false;
    const uint32_t avail = lane < kWarps ? *(volatile uint32_t *)&sh->slot[lane].legal0 : 0u;
    uint32_t m = __ballot_sync(kFull, avail != 0);
    if (urgent_only) {
        m &= *(volatile uint32_t *)&sh->urgent;
        if (m == 0) return 0u;
    } else if (m == 0) {
        done = __shfl_sync(kFull, *(volatile int32_t *)&sh->active, 0) <= 0;
        if (!done) __nanosleep(200);
        return 0u;
    }
    vw = lowest_bit(m);
    StealSlot *vs = &sh->slot[vw];
    uint32_t bit = 0;
    if (lane == 0) {
        const uint32_t old = *(volatile uint32_t *)&vs->legal0;
        if (old) {
            const uint32_t high = 1u << highest_bit(old);
            atomicAdd(&vs->pending, 1);                           // before the take: the owner cannot finish under us
            if (atomicCAS(&vs->legal0, old, old & ~high) == old) bit = high;
            else atomicSub(&vs->pending, 1);
        }
    }
    bit = __shfl_sync(kFull, bit, 0);
    if (bit == 0) return 0u;
    __threadfence_block();
    const int b = (int)*(volatile int8_t *)&vs->root[lane];
    const uint32_t meta = *(volatile uint32_t *)&vs->meta;
    root = lane < 28 ? b : 0;
    player = (int)(meta & 1u);
    die = (int)(meta >> 8);
    return bit;
}

template <int kWarps>
__device__ __forceinline__ void deliver_child(StealShared<kWarps> *sh, StealResult *cta_results, int vw, const Choice &c, int lane)
{
    StealSlot *vs = &sh->slot[vw];
    uint32_t idx = 0;
    if (lane == 0) idx = atomicAdd(&vs->nres, 1u);
    idx = __shfl_sync(kFull, idx, 0);
    StealResult *r = cta_results + vw * kStealMaxResults + idx;
    r->v[lane] = (int8_t)c.v;
    if (lane == 0) {
        r->value = c.value; r->any = c.any ? 1 : 0; r->n_seq = c.n_seq; r->n_scored = c.n_scored;
        r->n_visited = c.n_visited; r->origin = (int)(c.moves & 31u); r->moves = c.moves;   // the stolen origin's code
    }
    __threadfence_block();
    __syncwarp();
    if (lane == 0) atomicSub(&vs->pending, 1);
    __syncwarp();                        // the caller's loop continues from here: reconverged (see k_selfplay)
}

// greedy or exploring ply; kExplore = false compiles the epsilon path out (smaller, fewer registers)
template <int kSets, bool kExplore>
__device__ __forceinline__ Choice choose_ply_fast(int root, int lane, int player, int d1, int d2, const PlyEvaluator &ev,
                                                  PlyCache<kSets> &cache, bool explore, uint32_t u,
                                                  uint32_t root_only = kFull, const ShareCtx *share = nullptr,
                                                  int4 *zstash = nullptr, bool carry = false)
{
    if (kExplore && explore) {
        CountLeaf cnt;
        walk_turn(root, lane, player, d1, d2, cnt);
        Choice c;
        c.v = root; c.moves = 0; c.value = __int_as_float(0x7fc00000); c.n_seq = cnt.n; c.n_scored = 0; c.n_visited = 0; c.any = cnt.n > 0;
        c.z_ok = false;
        if (cnt.n > 0) {
            PickLeaf pick((int)mulhi32(u, (uint32_t)cnt.n));
            walk_turn(root, lane, player, d1, d2, pick);
            c.v = pick.v;
            c.moves = pick.moves;
        }
        return c;
    }
    return greedy_ply<kSets>(root, lane, player, d1, d2, ev, cache, root_only, share, zstash, carry);
}

} // namespace bgx
