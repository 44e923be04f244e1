"""Variance-reduced rollouts (DESIGN 7e) restated from pinned pieces.  TEST INFRASTRUCTURE.

`rollout_vr` is `rollout_ref.rollout` (same lockstep loop, dice, outcome classes and reduction) plus the luck of every trial: at each
ply k < vr_plies of a live trial it values the mover's 21 rolls through the same greedy-ply and value functions (two-ply's reply
rule), forms E_k, luck_k and the trial's sum in the spec's order, all in float64, and reduces y_t = x_t - luck_t as the spec reduces
x_t.  With `rollout_ref.engine_ply(eng)` it is a bit-exact reference for the fused kernel, with `oracle_ply` one for the CPU oracle.
"""
import numpy as np

from rollout_ref import MAX_PLIES, dice, outcome_class, reduce_trials

# the 21 rolls in two-ply's order (a = 1..6, b = 1..a) and their weights out of 36
ROLL_A = np.array([a for a in range(1, 7) for b in range(1, a + 1)], np.int8)
ROLL_B = np.array([b for a in range(1, 7) for b in range(1, a + 1)], np.int8)
WEIGHT = np.where(ROLL_A == ROLL_B, 1.0, 2.0)


def roll_index(d1, d2):
    """index of the unordered roll (max, min) in the 21-roll list"""
    hi, lo = np.maximum(d1, d2).astype(np.int64), np.minimum(d1, d2).astype(np.int64)
    return hi * (hi - 1) // 2 + lo - 1


def roll_values(ply_fn, value_fn, states, movers):
    """L[m, 21]: the value the greedy ply reports for each roll of (state, mover), V(state, mover) where it has no sequence"""
    m = len(states)
    q = np.zeros((m * 21, 32), np.int8)
    q[:, :28] = np.repeat(states, 21, axis=0)
    q[:, 28] = np.repeat(movers, 21)
    q[:, 29] = np.tile(ROLL_A, m)
    q[:, 30] = np.tile(ROLL_B, m)
    _, val, anyseq = ply_fn(q)
    L = np.asarray(val, np.float32).copy()
    blocked = ~np.asarray(anyseq, bool)
    if blocked.any():
        rows = np.unique(np.flatnonzero(blocked) // 21)
        V = value_fn(states[rows], movers[rows])
        Vrow = np.zeros(m, np.float32)
        Vrow[rows] = V
        L[blocked] = Vrow[np.flatnonzero(blocked) // 21]
    return L.reshape(m, 21)


def expectation(L):
    """E[m] = sum(weight x L) / 36 in roll order, float64, not rounded"""
    acc = np.zeros(len(L), np.float64)
    for r in range(21):
        acc = acc + WEIGHT[r] * L[:, r].astype(np.float64)
    return acc / 36.0


def rollout_vr(ply_fn, value_fn, positions, trials, max_plies=0, vr_plies=MAX_PLIES, seed=0x5EED2026, stratify=True, on_vr_ply=None):
    """The spec, in lockstep.  -> rollout_ref.rollout's dict plus vr_mean f64[n], vr_std_err f64[n], trial_luck f64[n, T].
    on_vr_ply(item, ply, L, E, luck), if given, sees every VR ply (item indices into the flattened n x T trials)."""
    positions = np.asarray(positions, np.int8).reshape(-1, 32)
    n = len(positions)
    items = n * trials
    state = np.repeat(positions[:, :28], trials, axis=0).astype(np.int8)
    mover = np.repeat((positions[:, 28] != 0).astype(np.int8), trials)
    t = np.tile(np.arange(trials, dtype=np.int64), n)
    ply = np.zeros(items, np.int32)
    value = np.zeros(items, np.float32)
    outcome = np.zeros(items, np.int8)
    luck = np.zeros(items, np.float64)
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
        vr = ply[idx] < vr_plies
        if vr.any():
            j = np.flatnonzero(vr)
            L = roll_values(ply_fn, value_fn, q[j, :28], q[j, 28])
            E = expectation(L)
            Lp = L[np.arange(len(j)), roll_index(q[j, 29], q[j, 30])].astype(np.float64)
            luck_k = Lp - E
            luck[idx[j]] = luck[idx[j]] + luck_k
            if on_vr_ply is not None:
                on_vr_ply(idx[j], ply[idx[j]].copy(), L, E, luck_k)
        after, val, anyseq = ply_fn(q)
        after = np.asarray(after, np.int8)
        played = ply[idx] + 1
        won1 = after[:, 26] == 15
        won2 = ~won1 & (after[:, 27] == 15)
        cut = ~won1 & ~won2 & (played >= cap)
        x = np.asarray(val, np.float32).copy()
        blocked = cut & ~np.asarray(anyseq, bool)
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
           "trial_plies": ply.reshape(n, trials), "trial_luck": luck.reshape(n, trials), "mean": np.zeros(n), "std_err": np.zeros(n),
           "counts": np.zeros((n, 8), np.int64), "vr_mean": np.zeros(n), "vr_std_err": np.zeros(n)}
    for p in range(n):
        x, o, k = out["trial_value"][p], out["trial_outcome"][p], out["trial_plies"][p]
        out["mean"][p], out["std_err"][p], out["counts"][p] = reduce_trials(x, o, k)
        y = x.astype(np.float64) - out["trial_luck"][p]
        out["vr_mean"][p], out["vr_std_err"][p], _ = reduce_trials(y, o, k)
    return out
