"""Rollouts (DESIGN 7d) restated from pinned pieces.  TEST INFRASTRUCTURE.

`rollout` plays every trial of every position in lockstep, one ply per iteration, through a greedy-ply function and a value
function it is given, and reduces with the spec's sequential float64 sums.  Two instantiations:
  * `oracle_ply(orc, weights)`: the CPU oracle's greedy ply (`Oracle.greedy_batch`) and `Oracle.forward`;
  * `engine_ply(eng)`: the engine's own one-ply kernel (`BatchEngine.select_moves_host`) and `evaluate_host`, advanced here in
    Python.  Values are pure functions of the query (DESIGN 2.1-1), so this is a bit-exact reference for the fused rollout kernel.
Dice come from a numpy Philox4x32-10 that `philox_np` restates and a CPU test pins to `Oracle.philox`.
"""
import math
import os

import numpy as np

STREAM = 4                 # Philox stream of the rollout dice
MAX_PLIES = 4096           # BGX_ROLLOUT_MAX_PLIES

_M0, _M1, _W0, _W1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57), 0x9E3779B9, 0xBB67AE85
_MASK = np.uint64(0xFFFFFFFF)


def philox_np(seed, c0, c1, c2, c3):
    """Philox4x32-10 (bgx_core.h philox4x32_10) on arrays of counters -> (x0, x1, x2, x3) uint64 arrays of 32-bit words"""
    c = [np.asarray(x, np.uint64) & _MASK for x in np.broadcast_arrays(c0, c1, c2, c3)]
    k0, k1 = seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF
    for _ in range(10):
        p0, p1 = _M0 * c[0], _M1 * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ np.uint64(k0), p1 & _MASK, (p0 >> np.uint64(32)) ^ c[3] ^ np.uint64(k1), p0 & _MASK]
        k0, k1 = (k0 + _W0) & 0xFFFFFFFF, (k1 + _W1) & 0xFFFFFFFF
    return c


def die_np(x):
    """die_of: 1 + (x * 6) >> 32"""
    return (1 + ((np.asarray(x, np.uint64) * np.uint64(6)) >> np.uint64(32))).astype(np.int8)


def dice(seed, t, k, stratify):
    """Dice of ply k of trials t (arrays): the stratified first roll, else Philox(seed; k, t lo, t hi, 4)."""
    t = np.asarray(t, np.int64)
    k = np.broadcast_to(np.asarray(k, np.int64), t.shape)
    x = philox_np(seed, k, t & 0xFFFFFFFF, t >> 32, np.full(t.shape, STREAM))
    d1, d2 = die_np(x[0]), die_np(x[1])
    if stratify:
        first = k == 0
        r = t % 36
        d1 = np.where(first, 1 + r // 6, d1).astype(np.int8)
        d2 = np.where(first, 1 + r % 6, d2).astype(np.int8)
    return d1, d2


def outcome_class(s):
    """Outcome class of a final board (int[28]): 1 / 2 / 3 PLAYER1 single / gammon / backgammon, 4 / 5 / 6 PLAYER2, 0 not over."""
    s = np.asarray(s, np.int64)
    if s[26] == 15:
        loser_off, loser_bar, in_home, base = s[27], s[25], (s[18:24] < 0).any(), 0
    elif s[27] == 15:
        loser_off, loser_bar, in_home, base = s[26], s[24], (s[0:6] > 0).any(), 3
    else:
        return 0
    return base + (1 if loser_off else (3 if loser_bar or in_home else 2))


def reduce_trials(x, outcome, plies):
    """mean, std_err, counts[8] of one position from its per-trial arrays, float64 sums in trial order"""
    trials = len(x)
    acc = 0.0
    for v in x:
        acc += float(v)
    mean = acc / trials
    ss = 0.0
    for v in x:
        d = float(v) - mean
        ss += d * d
    se = math.sqrt(ss / (trials * (trials - 1))) if trials > 1 else math.nan
    counts = np.zeros(8, np.int64)
    for k in range(1, 7):
        counts[k - 1] = int((outcome == k).sum())
    counts[6] = int((outcome == 0).sum())
    counts[7] = int(np.asarray(plies, np.int64).sum())
    return mean, se, counts


def oracle_ply(orc, weights):
    def ply(q):
        g = orc.greedy_batch(weights, q, threads=(os.cpu_count() or 1) if len(q) >= 64 else 1)
        return g["after"], g["value"], g["n_seq"] > 0

    def value(states, movers):
        V = np.zeros(len(states), np.float32)
        for t in (0, 1):
            m = movers == t
            if m.any():
                V[m] = orc.forward(weights, orc.encode(np.asarray(states, np.int32)[m], t))
        return V
    return ply, value


def engine_ply(eng):
    def ply(q):
        o = eng.select_moves_host(q)
        return o["chosen"][:, :28], o["value"], o["n_seq"] > 0

    def value(states, movers):
        r = np.zeros((len(states), 32), np.int8)
        r[:, :28] = states
        r[:, 28] = movers
        return eng.evaluate_host(r)
    return ply, value


def rollout(ply_fn, value_fn, positions, trials, max_plies=0, seed=0x5EED2026, stratify=True, on_ply=None):
    """The spec, in lockstep.  -> dict(mean f64[n], std_err f64[n], counts int64[n,8], trial_value f32[n,T], trial_outcome
    int8[n,T], trial_plies int32[n,T]).  on_ply(queries, after, value, any), if given, sees every ply played."""
    positions = np.asarray(positions, np.int8).reshape(-1, 32)
    n = len(positions)
    items = n * trials
    state = np.repeat(positions[:, :28], trials, axis=0).astype(np.int8)
    mover = np.repeat((positions[:, 28] != 0).astype(np.int8), trials)
    t = np.tile(np.arange(trials, dtype=np.int64), n)
    ply = np.zeros(items, np.int32)
    value = np.zeros(items, np.float32)
    outcome = np.zeros(items, np.int8)
    cap = max_plies if max_plies > 0 else MAX_PLIES
    active = np.ones(items, bool)
    for i in np.flatnonzero((state[:, 26] == 15) | (state[:, 27] == 15)):       # over already: ends at ply 0
        value[i] = 1.0 if state[i, 26] == 15 else 0.0
        outcome[i] = outcome_class(state[i])
        active[i] = False
    while active.any():
        idx = np.flatnonzero(active)
        q = np.zeros((len(idx), 32), np.int8)
        q[:, :28] = state[idx]
        q[:, 28] = mover[idx]
        q[:, 29], q[:, 30] = dice(seed, t[idx], ply[idx], stratify)
        after, val, anyseq = ply_fn(q)
        after = np.asarray(after, np.int8)
        if on_ply is not None:
            on_ply(q, after, val, anyseq)
        played = ply[idx] + 1
        won1 = after[:, 26] == 15
        won2 = ~won1 & (after[:, 27] == 15)
        cut = ~won1 & ~won2 & (played >= cap)
        x = np.asarray(val, np.float32).copy()
        blocked = cut & ~anyseq
        if blocked.any():
            x[blocked] = value_fn(q[blocked, :28], q[blocked, 28])
        done = won1 | won2 | cut
        for j in np.flatnonzero(done):
            i = idx[j]
            value[i] = 1.0 if won1[j] else (0.0 if won2[j] else x[j])
            outcome[i] = outcome_class(after[j]) if not cut[j] else 0
            active[i] = False
        state[idx] = after
        ply[idx] = played
        mover[idx] ^= 1
    out = {"trial_value": value.reshape(n, trials), "trial_outcome": outcome.reshape(n, trials),
           "trial_plies": ply.reshape(n, trials), "mean": np.zeros(n), "std_err": np.zeros(n), "counts": np.zeros((n, 8), np.int64)}
    for p in range(n):
        out["mean"][p], out["std_err"][p], out["counts"][p] = reduce_trials(out["trial_value"][p], out["trial_outcome"][p],
                                                                            out["trial_plies"][p])
    return out
