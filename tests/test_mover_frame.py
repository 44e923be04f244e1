"""The greedy walk runs in the mover's frame (DESIGN 2.1-20): for PLAYER2 the points are negated and the bar and borne-off
lanes swapped at the start of a ply, and the chosen afterstate is converted back at its end.  These tests pin what the frame
touches, for both movers, on positions built to reach each of its edges:
  - the mover on the bar, entering and blocked;
  - hits that send a blot to the enemy's bar;
  - exact bear-off and both over-bear quirks (SURVEY A.3 Q3/Q4);
  - sequences that end early, at depths 0-3 in doubles and 0-1 in non-doubles (the out-of-line early-leaf scorer);
  - big doubles walked by several warps (the sharing protocol publishes and merges positions).
Every position is there twice, once per mover: the second copy is the first seen from the other side of the board (not the
same turn: the over-bear rules differ between the players)."""
import numpy as np
import pytest

from conftest import golden_weights
from test_ply_exactness import assert_same, check_integer_rule, integer_rule, restart_loop_matches_population, tie_net

KEYS = ("chosen", "moves", "moves_len", "value", "n_seq")


def mirrored(q):
    """The same positions with the other player to move: point i <-> 23 - i with the colours swapped, bars and borne-off
    counts swapped.  Dice stay."""
    m = q.copy()
    m[:, :24] = -q[:, 23::-1]
    m[:, 24], m[:, 25] = q[:, 25], q[:, 24]
    m[:, 26], m[:, 27] = q[:, 27], q[:, 26]
    m[:, 28] = 1 - q[:, 28]
    return m


def record(points, bar=(0, 0), off=(0, 0), d1=1, d2=1):
    """A PLAYER1-to-move record from {point index: count} (+ PLAYER1, - PLAYER2)."""
    r = np.zeros(32, np.int8)
    for i, c in points.items():
        r[i] = c
    r[24], r[25] = bar
    r[26], r[27] = off
    r[29], r[30] = d1, d2
    return r


def built():
    """Hand-made PLAYER1 positions for the edges random positions reach rarely, under every roll."""
    closed = {i: -2 for i in range(6)}                    # PLAYER2's home board closed against PLAYER1's entry
    base = [
        record({**closed, 12: 2, 18: 3}, bar=(1, 0), off=(0, 0)),                       # on the bar, blocked
        record({0: -2, 1: -2, 2: -2, 3: -2, 4: -2, 12: 2, 18: 2}, bar=(2, 0)),         # one entry point open
        record({0: -2, 2: -1, 4: -1, 10: 3, 20: 2}, bar=(1, 0)),                        # enter with a hit
        record({18: 1, 19: -1, 20: 1, 21: -1, 22: 2, 23: -1, 5: -2}, bar=(0, 1)),      # blots around the mover
        record({23: 2, 22: 3, 20: 2}, off=(8, 0)),                                      # bear-off from the low home points
        record({18: 2, 19: 1, 21: 3}, off=(9, 2)),                                      # over-bear from the highest point
        record({21: 1, 23: 1, 0: -3, 3: -2}, off=(13, 10)),                             # two checkers left
        record({19: 4, 20: 4, 18: 2, 6: -2, 7: -2, 8: -2, 9: -2}, off=(5, 0)),          # doubles that run out of moves
        record({17: 1, 19: 2, 20: -2, 21: -2, 22: -2, 23: -2, 15: -2, 16: -2}, off=(10, 0)),   # one checker outside, walled in
    ]
    out = []
    for r in base:
        for d1 in range(1, 7):
            for d2 in range(1, 7):
                x = r.copy()
                x[29], x[30] = d1, d2
                out.append(x)
    return np.array(out)


@pytest.fixture(scope="module")
def frame_queries():
    from bgx.synth import make_queries
    q, _ = make_queries(6000, seed=2204)
    q = np.concatenate([q, built()])
    return np.concatenate([q, mirrored(q)])


def coverage(orc, q):
    """-> {edge: number of queries that reach it} from the oracle's sequence lists, per mover."""
    cov = {}

    def add(k):
        cov[k] = cov.get(k, 0) + 1

    for r in q:
        p, d1, d2 = int(r[28]), int(r[29]), int(r[30])
        s = r[:28].astype(np.int32)
        mv, ln, st = orc.turn_sequences(s, p, d1, d2)
        dbl = d1 == d2
        full = 4 if dbl else 2
        if s[24 + p] > 0:
            add((p, "bar blocked" if len(ln) == 0 or max(ln) == 0 else "bar entering"))
        if len(ln) == 0:
            add((p, "no sequence", dbl))
            continue
        if len(ln) and (st[:, 25 - p] > s[25 - p]).any():
            add((p, "hit"))
        for L in set(int(x) for x in ln):
            if L < full:
                add((p, "early", dbl, L))
        if len(ln) > 500 and dbl:
            add((p, "big double"))
        target = 25 if p == 0 else 0
        for j in range(len(ln)):
            for o, d in mv[j, :ln[j]]:
                if d == target and o not in (0, 25):
                    dist = abs(target - int(o))
                    if dist in (d1, d2):
                        add((p, "exact bear-off"))
                    elif dist < min(d1, d2):
                        add((p, "over-bear"))
    return cov


def test_frame_queries_reach_every_edge(orc, frame_queries):
    cov = coverage(orc, frame_queries)
    for p in (0, 1):
        for k in ("bar entering", "bar blocked", "hit", "exact bear-off", "over-bear", "big double"):
            assert cov.get((p, k), 0) >= 10, (p, k, cov.get((p, k), 0))
        for L in range(4):
            assert cov.get((p, "early", True, L), 0) >= 5, (p, "double ends at depth", L, cov)
        assert cov.get((p, "early", False, 1), 0) >= 5, (p, "non-double ends at depth 1", cov)
        assert cov.get((p, "no sequence", False), 0) + cov.get((p, "early", True, 0), 0) >= 5, (p, "no move at all", cov)


# ------------------------------------------------------------------ GPU

@pytest.fixture(scope="module")
def eng():
    from bgx.engine import BatchEngine
    e = BatchEngine(0)
    yield e
    e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["off", "bar"])
def test_select_moves_in_both_frames_is_the_integer_rule(eng, orc, frame_queries, kind):
    """Under a tie net the pick is an integer fact about the enumeration: afterstate, sequence and N equal the oracle's for both
    movers, V is the float64 forward's within 1e-5 and, bit for bit, the evaluator's value of the afterstate it reports."""
    w = tie_net(kind)
    eng.set_weights(*w)
    out = eng.select_moves_host(frame_queries)
    check_integer_rule(orc, w, frame_queries, out, integer_rule(orc, frame_queries, (kind,)), kind)
    has = out["n_seq"] > 0
    assert np.array_equal(eng.evaluate_host(out["chosen"][has]).view(np.uint32), out["value"][has].view(np.uint32))


@pytest.mark.gpu
def test_select_moves_in_both_frames_vs_oracle(eng, orc, golden, frame_queries):
    """The trained net: N and the moves of every pick are the oracle's except where two afterstates' values agree to 1e-5 (the
    oracle sums in float, the kernels in fixed point); V is the evaluator's value of the chosen afterstate bit for bit."""
    w = golden_weights(golden("model.npz"), "trained")
    eng.set_weights(*w)
    q = frame_queries
    out = eng.select_moves_host(q)
    ref = orc.greedy_batch(w, q)
    assert np.array_equal(out["n_seq"].astype(np.int64), ref["n_seq"])
    has = ref["n_seq"] > 0
    assert np.array_equal(out["chosen"][~has, :28], q[~has, :28]) and np.isnan(out["value"][~has]).all()
    assert np.array_equal(eng.evaluate_host(out["chosen"][has]).view(np.uint32), out["value"][has].view(np.uint32))
    same = (out["chosen"][:, :28] == ref["after"]).all(1)
    diff = np.flatnonzero(has & ~same)
    assert diff.size <= 0.005 * has.sum(), diff.size
    for t in (0, 1):
        idx = diff[q[diff, 28] == t]
        if idx.size:
            v = orc.forward(w, orc.encode(out["chosen"][idx, :28].astype(np.int32), t))
            assert (np.abs(v - ref["value"][idx]) <= 1e-5 * np.abs(ref["value"][idx])).all()
    ok = has & same
    assert np.array_equal(out["moves_len"][ok], ref["moves_len"][ok])
    assert (out["moves"][ok] == ref["moves"][ok]).reshape(ok.sum(), -1).all()


@pytest.mark.gpu
@pytest.mark.parametrize("net", ["trained", "bar"])
def test_shared_doubles_in_both_frames(golden, frame_queries, net):
    """Every double of the set with its CTA helping at once (giant threshold at the publishing threshold): helpers walk stolen
    sub-trees from the published root and the owner merges; the result is the default engine's bit for bit."""
    from bgx.engine import BatchEngine
    w = golden_weights(golden("model.npz"), net) if net == "trained" else tie_net(net)
    dbl = frame_queries[frame_queries[:, 29] == frame_queries[:, 30]]
    a, b = BatchEngine(0), BatchEngine(0)
    try:
        a.set_weights(*w)
        b.set_weights(*w)
        b.set_option("select_giant_min", 4)                   # kStealMinChildren
        assert_same(b.select_moves_host(dbl), a.select_moves_host(dbl), KEYS, what=net)
        big = dbl[a.select_moves_host(dbl)["n_seq"] > 500][:64]     # alone on the GPU: every sub-tree that can be taken is
        assert len(big) == 64
        assert_same(a.select_moves_host(big), b.select_moves_host(big), KEYS, what=net + " alone")
    finally:
        a.close()
        b.close()


@pytest.mark.gpu
def test_selfplay_step_in_both_frames_is_the_host_driven_loop(eng, golden):
    """k_selfplay carries the chosen afterstate, the game-over test and the root pre-activation from ply to ply in the real
    frame: 400 plies of 1,500 slots (games through contact, the bar and the bear-off, both movers) equal the host-driven loop of
    k_select launches bit for bit."""
    eng.set_weights(*golden_weights(golden("model.npz"), "trained"))
    st = restart_loop_matches_population(eng, 1500, 400)
    assert st["games_finished"] > 3 * 1500
