"""Two-ply move selection (DESIGN 7c) restated on the CPU checkers.  TEST INFRASTRUCTURE.

Built only from pieces that are already pinned to the reference: `Oracle.turn_sequences` for the candidates, the threaded
`Oracle.greedy_batch` for the opponent's replies, `Oracle.forward` for one-ply values and blocked replies, and a float64
combination of the reply values in the fixed roll order.
"""
import numpy as np

ROLLS = [(a, b) for a in range(1, 7) for b in range(1, a + 1)]        # a = 1..6, b = 1..a
WEIGHTS = np.array([1.0 if a == b else 2.0 for a, b in ROLLS])         # of 36


def candidates(orc, rec):
    """Distinct afterstates of a query in order of first appearance -> (states int32[U,28], moves int8[U,4,2], lens int8[U])."""
    mv, ln, st = orc.turn_sequences(rec[:28].astype(np.int32), int(rec[28]), int(rec[29]), int(rec[30]))
    first = {}
    for i in range(len(ln)):
        first.setdefault(st[i].tobytes(), i)
    idx = np.array(sorted(first.values()), np.int64)
    return st[idx], mv[idx], ln[idx]


def expanded_mask(v1, wins, player, K):
    """Which candidates get the 21 replies: none if one wins, else all (K = 0 or K >= U) or the K best one-ply values for the
    mover, first appearance on ties."""
    U = len(v1)
    if U == 0 or wins.any():
        return np.zeros(U, bool)
    if K == 0 or K >= U:
        return np.ones(U, bool)
    key = -v1 if player else v1
    best = sorted(range(U), key=lambda i: (-key[i], i))[:K]
    m = np.zeros(U, bool)
    m[best] = True
    return m


def pick(e2, expanded, wins, player):
    """-> (index or -1, value): the first winning candidate, else the first arg-max (PLAYER1) / arg-min (PLAYER2) of E2."""
    if len(e2) == 0:
        return -1, np.float32(np.nan)
    if wins.any():
        return int(np.argmax(wins)), np.float32(0.0 if player else 1.0)
    key = np.where(expanded, -e2 if player else e2, -np.inf)
    i = int(np.argmax(key))
    return i, e2[i]


def combine(R):
    """E2 from the 21 reply values in roll order: float64 sum, rounded once to fp32."""
    acc = 0.0
    for w, r in zip(WEIGHTS, R):
        acc += w * float(r)
    return np.float32(acc / 36.0)


def twoply_batch(orc, weights, records, max_candidates=0):
    """Per query a dict: states int32[U,28], moves int8[U,4,2], lens int8[U] (first sequence of every candidate), v1 f32[U]
    (one-ply value for the mover), wins bool[U], expanded bool[U], e2 f32[U] (NaN where not expanded), pick (-1: no
    candidate), value, n_expanded."""
    records = np.asarray(records, np.int8).reshape(-1, 32)
    out, replies, owner = [], [], []
    for q, rec in enumerate(records):
        p = int(rec[28])
        st, mv, ln = candidates(orc, rec)
        U = len(ln)
        v1 = orc.forward(weights, orc.encode(st, p)) if U else np.zeros(0, np.float32)
        wins = st[:, 26 + p] == 15 if U else np.zeros(0, bool)
        exp = expanded_mask(v1, wins, p, max_candidates)
        out.append({"states": st, "moves": mv, "lens": ln, "v1": v1, "wins": wins, "expanded": exp,
                    "e2": np.full(U, np.nan, np.float32)})
        for i in np.flatnonzero(exp):
            r = np.zeros((len(ROLLS), 32), np.int8)
            r[:, :28] = st[i]
            r[:, 28] = 1 - p
            r[:, 29:31] = ROLLS
            replies.append(r)
            owner.append((q, i))
    if replies:
        rr = np.concatenate(replies)
        g = orc.greedy_batch(weights, rr)
        R = g["value"].astype(np.float32).copy()
        still = g["moves_len"] == 0                              # no move for the opponent: the position keeps V(A, opponent)
        for t in (0, 1):
            m = still & (rr[:, 28] == t)
            if m.any():
                R[m] = orc.forward(weights, orc.encode(rr[m, :28].astype(np.int32), t))
        for k, (q, i) in enumerate(owner):
            out[q]["e2"][i] = combine(R[k * len(ROLLS):(k + 1) * len(ROLLS)])
    for q, rec in enumerate(records):
        o = out[q]
        o["pick"], o["value"] = pick(o["e2"], o["expanded"], o["wins"], int(rec[28]))
        o["n_expanded"] = int(o["expanded"].sum())
    return out
