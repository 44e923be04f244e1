"""GPU parity tests: every batched C-ABI entry point of libbgx against the reference's golden
vectors and the CPU oracle on the same seeded inputs.  Integer results (move sets, order,
boards, bar/off counts, winners, encodings) must be bit-exact; values and TD updates must be
within 1e-5 relative (BASELINE.json north_star)."""
import hashlib

import numpy as np
import pytest

from conftest import golden_weights

pytestmark = pytest.mark.gpu

SEED = 0x5EED2026
START_BOARD_NP = np.array([2, 0, 0, 0, 0, -5, 0, -3, 0, 0, 0, 5, -5, 0, 0, 0, 3, 0, 5, 0, 0, 0, 0, -2], np.int8)   # game.cpp:251


@pytest.fixture(scope="module")
def eng():
    from bgx.engine import BatchEngine
    e = BatchEngine(0)
    yield e
    e.close()


def records_from(states, player, dice=None):
    st = np.asarray(states)
    r = np.zeros((st.shape[0], 32), np.int8)
    r[:, :28] = st[:, :28]
    r[:, 28] = player
    if dice is not None:
        r[:, 29:31] = dice
    return r


# ------------------------------------------------------------------ enumeration (bit-exact)

def test_enumerate_summary_golden(eng, golden):
    g = golden("enum_summary.npz")
    n, u, d = eng.enumerate_summary_host(g["queries"])
    assert np.array_equal(n, g["n_seq"])
    assert np.array_equal(u, g["n_unique"])
    assert np.array_equal(d, g["digest"])


def test_enumerate_full_golden(eng, golden):
    g = golden("enum_full.npz")
    offsets, mv, ln, st = eng.enumerate_host(g["queries"])
    assert np.array_equal(offsets, g["offsets"])
    assert np.array_equal(mv.reshape(-1, 8), g["moves"])
    assert np.array_equal(ln, g["lens"])
    assert np.array_equal(st[:, :28], g["states"])
    mover = np.repeat(g["queries"][:, 28], np.diff(g["offsets"]))
    assert np.array_equal(st[:, 28], mover)


def test_enumerate_edge_cases(eng, orc):
    from bgx.synth import start_record
    # empty batch
    n, u, d = eng.enumerate_summary_host(np.zeros((0, 32), np.int8))
    assert len(n) == 0
    offsets, mv, ln, st = eng.enumerate_host(np.zeros((0, 32), np.int8))
    assert offsets.tolist() == [0] and len(ln) == 0
    # blocked: non-double -> 0 sequences; double -> one empty sequence (quirk Q5)
    blocked = np.zeros((2, 32), np.int8)
    blocked[:, :6] = -2
    blocked[:, 24] = 1
    blocked[:, 26] = 14
    blocked[:, 27] = 3
    blocked[0, 29:31] = (3, 4)
    blocked[1, 29:31] = (3, 3)
    n, u, d = eng.enumerate_summary_host(blocked)
    assert n.tolist() == [0, 1] and u.tolist() == [0, 1]
    offsets, mv, ln, st = eng.enumerate_host(blocked)
    assert offsets.tolist() == [0, 0, 1] and ln.tolist() == [0]
    assert np.array_equal(st[0, :28], blocked[1, :28])
    # the heaviest opening roll (2-2: 538 sequences) and a single ragged batch of 3
    q = np.stack([start_record(0, 2, 2), start_record(1, 6, 5), start_record(0, 3, 3)])
    n, u, d = eng.enumerate_summary_host(q)
    assert n.tolist() == [538, 14, 536] and u.tolist() == [75, 7, 73]


def test_enumerate_vs_oracle_fresh_seed(eng, orc):
    from bgx.synth import make_queries
    q, _ = make_queries(30000, seed=424242)
    n, u, d = eng.enumerate_summary_host(q)
    for i in range(0, len(q), 7):                      # every 7th query: ~4.3k oracle enumerations
        r = q[i]
        assert orc.turn_summary(r[:28].astype(np.int32), r[28], r[29], r[30]) == (int(n[i]), int(u[i]), int(d[i])), i
    # ordered lists for a slice, against the oracle
    sub = q[:600]
    offsets, mv, ln, st = eng.enumerate_host(sub)
    for i, r in enumerate(sub):
        omv, oln, ost = orc.turn_sequences(r[:28].astype(np.int32), r[28], r[29], r[30])
        a, b = offsets[i], offsets[i + 1]
        assert np.array_equal(mv[a:b], omv) and np.array_equal(ln[a:b], oln)
        assert np.array_equal(st[a:b, :28], ost.astype(np.int8))


def test_enumerate_million_position_properties(eng):
    """BASELINE configs[1] at full size: 10^6 seeded positions.  Size-independent properties:
    swapping the dice permutes the sequence list (same N, same U, different order => different
    digest unless N <= 1), doubles never emit more than 4 moves, and the run is deterministic."""
    from bgx.synth import make_queries
    q, _ = make_queries(1_000_000, seed=20260101)
    n, u, d = eng.enumerate_summary_host(q)
    sw = q.copy()
    sw[:, 29], sw[:, 30] = q[:, 30], q[:, 29]
    n2, u2, d2 = eng.enumerate_summary_host(sw)
    assert np.array_equal(n, n2) and np.array_equal(u, u2)
    dbl = q[:, 29] == q[:, 30]
    assert np.array_equal(d[dbl], d2[dbl])
    assert (u >= 0).all() and (u <= n).all() and ((n == 0) == (u == 0)).all()
    n3, u3, d3 = eng.enumerate_summary_host(q)
    assert np.array_equal(n, n3) and np.array_equal(u, u3) and np.array_equal(d, d3)
    assert int(n.sum()) > 30_000_000


# The reference's sequence counts (int64) and ordered digests (uint64) on the 10^6-position sweep: their total and the
# sha256 of the two arrays' bytes, recorded by tests/golden/make_recorded.py sweep (provenance there).  Checked on every
# run; the reference engine itself is compared live as well where oracle/_ref holds it.
REF_SWEEP_SEQUENCES = 67_894_650
REF_SWEEP_SHA256 = "3db2f035a5ce23eef692c282c4f654340f44121340da094cbad69c2026c06709"


def test_enumerate_million_positions_bit_exact_vs_reference(eng, orc, golden):
    """BASELINE north_star: "bit-exact move sets against the reference on 10^6 seeded positions".
    The configs[1] sweep as SURVEY 8(d) config 2 defines it: 500,000 constructive positions + 500,000 positions
    sampled at uniform plies from random-vs-random playouts (config 1), dice over all 36 ordered pairs.  EVERY position:
    sequence count and the ordered digest (which pins every move of every sequence, its order and its resulting
    28-int state) against the UNMODIFIED reference engine's evaluateTurnSequences (game.cpp:193-222; ~68 M sequences):
    against its recorded results (REF_SWEEP_*), and live through oracle/_ref where that is built; and count, exact number of
    distinct afterstates and digest against the C oracle."""
    from bgx.synth import CLASSES, make_sweep_queries
    from oracle.oracle import RefHarness
    eng.set_weights(*golden_weights(golden("model.npz"), "rand"))
    q, cls = make_sweep_queries(eng, 1_000_000)
    play = q[cls == len(CLASSES)]
    assert len(play) == 500_000
    b = play[:, :24].astype(np.int64)
    assert np.array_equal(np.where(b > 0, b, 0).sum(1) + play[:, 24] + play[:, 26], np.full(len(play), 15))
    assert np.array_equal(np.where(b < 0, -b, 0).sum(1) + play[:, 25] + play[:, 27], np.full(len(play), 15))
    assert ((play[:, 29] >= 1) & (play[:, 29] <= 6) & (play[:, 30] >= 1) & (play[:, 30] <= 6)).all()
    assert len(np.unique(play, axis=0)) > 400_000                 # beyond the opening plies the playouts do not repeat
    n, u, d = eng.enumerate_summary_host(q)
    on, ou, od = orc.turn_summary_batch(q)
    assert np.array_equal(n.astype(np.int64), on)
    assert np.array_equal(u.astype(np.int64), ou)
    assert np.array_equal(d.astype(np.uint64), od)
    assert int(n.sum()) == REF_SWEEP_SEQUENCES
    assert hashlib.sha256(on.tobytes() + od.tobytes()).hexdigest() == REF_SWEEP_SHA256
    if not RefHarness.available():
        return
    rn, rd = RefHarness().turn_summary_batch(q)
    assert np.array_equal(n.astype(np.int64), rn)
    assert np.array_equal(d.astype(np.uint64), rd)


# ------------------------------------------------------------------ encoding (bit-exact) and values

def test_encode_golden_bit_exact(eng, golden):
    g = golden("model.npz")
    X = eng.encode_host(records_from(g["states"], g["turn"]))
    assert np.array_equal(X.view(np.uint32), g["X"].view(np.uint32))


@pytest.mark.parametrize("n", [1, 2, 3, 31, 32, 33, 1000, 65537])
def test_encode_ragged_sizes_vs_oracle(eng, orc, n):
    from bgx.synth import make_queries
    q, _ = make_queries(n, seed=n)
    X = eng.encode_host(q)
    for t in (0, 1):
        sel = q[:, 28] == t
        if sel.any():
            ref = orc.encode(q[sel, :28].astype(np.int32), t)
            assert np.array_equal(X[sel].view(np.uint32), ref.view(np.uint32))


@pytest.mark.parametrize("tag", ["rand", "trained"])
def test_values_golden(eng, golden, tag):
    g = golden("model.npz")
    eng.set_weights(*golden_weights(g, tag))
    V = eng.evaluate_host(records_from(g["states"], g["turn"]))
    ref = g[f"v_{tag}"]
    assert np.max(np.abs(V - ref) / np.abs(ref)) <= 1e-5
    got = eng.get_weights()
    for a, b in zip(got, golden_weights(g, tag)):
        assert np.array_equal(np.asarray(a).reshape(-1), np.asarray(b).reshape(-1))


@pytest.mark.parametrize("tag", ["trained", "rand"])
def test_values_hundred_thousand_afterstates(eng, orc, golden, tag):
    """SURVEY 8d config 3: value parity <= 1e-5 relative on a 10^5-afterstate sample - the afterstates the engine itself
    enumerates for 3,000 seeded sweep positions (mover's turn flag, model.py:139-140), scored by k_evaluate and by the
    oracle's dense fp32 forward (model.py:63-67)."""
    from bgx.synth import make_queries
    w = golden_weights(golden("model.npz"), tag)
    eng.set_weights(*w)
    q, _ = make_queries(3000, seed=4242)
    offsets, mv, ln, st = eng.enumerate_host(q)
    counts = np.diff(offsets)
    player = np.repeat(q[:, 28], counts)
    rows = records_from(st[:, :28], player)
    keep = np.random.default_rng(5).permutation(len(rows))[:100000]
    assert len(keep) == 100000
    rows = rows[keep]
    V = eng.evaluate_host(rows)
    ref = np.zeros(len(rows), np.float32)
    for pl in (0, 1):
        m = rows[:, 28] == pl
        ref[m] = orc.forward(w, orc.encode(rows[m, :28].astype(np.int32), pl))
    assert np.max(np.abs(V - ref) / np.abs(ref)) <= 1e-5
    X = eng.encode_host(rows[:20000])
    for pl in (0, 1):
        m = rows[:20000, 28] == pl
        assert np.array_equal(X[m], orc.encode(rows[:20000][m, :28].astype(np.int32), pl))


# ------------------------------------------------------------------ batched make_move

def check_choice(orc, w, rec, chosen, value=None, n_seq=None):
    """The engine's pick for one query is the oracle's, or differs only inside the 1e-5 value tolerance.
    Returns 1 for such a near-tie, 0 for an identical pick."""
    s = rec[:28].astype(np.int32)
    pl = int(rec[28])
    idx, after, v, n = orc.greedy_ply(w, s, pl, rec[29], rec[30])
    if n_seq is not None:
        assert n == n_seq
    got = chosen[:28].astype(np.int32)
    if idx < 0:
        assert np.array_equal(got, s) and chosen[31] == 0
        return 0
    assert chosen[28] == pl
    vg = v if np.array_equal(got, after) else orc.forward(w, orc.encode(got[None], pl))[0]
    if value is not None:
        assert abs(value - vg) <= 1e-5 * abs(vg)          # the reported value is the oracle's for that afterstate
    if np.array_equal(got, after):
        return 0
    assert abs(vg - v) <= 1e-5 * abs(v), "different afterstate outside the value tolerance"
    return 1


@pytest.mark.parametrize("tag", ["rand", "trained"])
def test_select_moves_vs_oracle(eng, orc, golden, tag):
    from bgx.synth import make_queries
    w = golden_weights(golden("model.npz"), tag)
    eng.set_weights(*w)
    q, _ = make_queries(3000, seed=31337)
    out = eng.select_moves_host(q)
    soft = 0
    for i, r in enumerate(q):
        soft += check_choice(orc, w, r, out["chosen"][i], out["value"][i], int(out["n_seq"][i]))
        # the reported sequence really leads to the reported afterstate
        s = r[:28].astype(np.int32)
        for j in range(out["moves_len"][i]):
            o, d = (int(x) for x in out["moves"][i, j])
            ok, _, s = orc.try_move(s, int(r[28]), abs(o - d), o, d)
            assert ok
        assert np.array_equal(s, out["chosen"][i, :28].astype(np.int32))
        assert 0 <= out["n_scored"][i] <= max(out["n_seq"][i], 0)
    assert soft <= (300 if tag == "rand" else 30), soft     # near-ties: ~10 % with random-init weights (SURVEY 7.3-3)


@pytest.mark.parametrize("tag", ["trained", "rand"])
def test_select_moves_large_sample_vs_oracle(eng, orc, golden, tag):
    """60,000 seeded positions (incl. bar entry, doubles, bear-off) per weight set against the threaded oracle: N exact everywhere;
    the chosen afterstate is the oracle's except inside the 1e-5 value tolerance; and wherever the afterstate is the oracle's, the
    REPORTED SEQUENCE is the oracle's too - the first one in reference order among all that lead there (model.py:212-220), which
    is what memoised doubles, twin leaves and shared sub-trees must not disturb."""
    from bgx.synth import make_queries
    w = golden_weights(golden("model.npz"), tag)
    eng.set_weights(*w)
    q, _ = make_queries(60000, seed=777)
    out = eng.select_moves_host(q)
    ref = orc.greedy_batch(w, q)
    assert np.array_equal(out["n_seq"].astype(np.int64), ref["n_seq"])
    has = ref["n_seq"] > 0
    same = (out["chosen"][:, :28] == ref["after"]).all(1)
    assert same[~has].all()                                   # no sequence: the position comes back unchanged
    diff = np.flatnonzero(has & ~same)
    if diff.size:                                             # near-ties: the engine's pick is worth the oracle's best within 1e-5
        for t in (0, 1):
            idx = diff[q[diff, 28] == t]
            if idx.size:
                v = orc.forward(w, orc.encode(out["chosen"][idx, :28].astype(np.int32), t))
                assert (np.abs(v - ref["value"][idx]) <= 1e-5 * np.abs(ref["value"][idx])).all()
    assert diff.size <= (0.12 if tag == "rand" else 0.012) * has.sum(), diff.size
    ok = has & same
    assert (np.abs(out["value"][ok] - ref["value"][ok]) <= 1e-5 * np.abs(ref["value"][ok])).all()
    exact = (out["moves"].reshape(-1, 8) == ref["moves"].reshape(-1, 8)).all(1) & (out["moves_len"] == ref["moves_len"])
    assert exact[ok].all(), (int((~exact[ok]).sum()), int(ok.sum()))


def test_sfu_approximations_are_monotone(eng):
    """The greedy ply ranks afterstates by the integer output sum and evaluates V = sigmoid(sum / Y + b2) only for a sum that
    beats the best so far (bgx_ply.cuh PlyEvaluator::value_of).  That is the reference's strict first-index arg-best over V
    (model.py:205-213) exactly if V is a non-decreasing function of the sum; the two SFU approximations in it carry no such
    guarantee on paper, so it is checked on the device, exhaustively (every neighbouring pair of finite floats)."""
    assert eng.sfu_monotone() == (0, 0)


@pytest.mark.parametrize("tag", ["rand", "trained"])
def test_select_moves_is_a_pure_function_of_the_query(eng, golden, tag):
    """The choice must not depend on batch composition, on which warp walked a position, on what the
    per-warp caches held, or on how many sub-trees of a big double were walked by helper warps: the
    same queries alone (most warps idle, heavy sharing), inside a large batch (little sharing), in a
    different order and through the asynchronous lanes give bit-identical records, moves and values."""
    import torch
    from bgx.synth import make_queries
    w = golden_weights(golden("model.npz"), tag)
    eng.set_weights(*w)
    q, _ = make_queries(20000, seed=424242)
    keys = ("chosen", "moves", "moves_len", "value", "n_seq")
    whole = eng.select_moves_host(q)
    big = np.flatnonzero((q[:, 29] == q[:, 30]) & (whole["n_seq"] > 500))[:64]      # big doubles
    assert big.size >= 16
    few = eng.select_moves_host(q[big])                                             # 64 queries on 2,368 warps
    for k in keys:
        assert np.array_equal(few[k], whole[k][big], equal_nan=(k == "value")), k
    perm = np.random.default_rng(1).permutation(q.shape[0])
    shuf = eng.select_moves_host(q[perm])
    for k in keys:
        assert np.array_equal(shuf[k], whole[k][perm], equal_nan=(k == "value")), k
    # asynchronous lanes: two halves in flight at once, pinned buffers
    h = q.shape[0] // 2
    pin = {k: torch.from_numpy(np.zeros_like(whole[k])).pin_memory().numpy() for k in keys}
    qp = torch.from_numpy(q.copy()).pin_memory().numpy()
    for lane, (lo, hi) in enumerate(((0, h), (h, q.shape[0]))):
        eng.select_moves_host_async(lane, qp[lo:hi], {k: pin[k][lo:hi] for k in keys})
    eng.wait(0)
    eng.wait(1)
    for k in keys:
        assert np.array_equal(pin[k], whole[k], equal_nan=(k == "value")), k
    # a lane holds one batch at a time
    from bgx.lib import BgxError
    eng.select_moves_host_async(2, qp[:16], {"chosen": pin["chosen"][:16]})
    with pytest.raises(BgxError):
        eng.select_moves_host_async(2, qp[:16], {"chosen": pin["chosen"][:16]})
    eng.wait(2)


def test_play_ply_is_select_plus_advance(eng, golden):
    """bgx_play_ply_host_async (one iteration of play_game's loop, train.py:103-121) = bgx_select_moves_host followed by
    bgx_advance_host, byte for byte, whatever the lane and the batch split."""
    from bgx import host as H
    from bgx.synth import make_queries
    eng.set_weights(*golden_weights(golden("model.npz"), "trained"))
    q, _ = make_queries(20000, seed=99)
    # a few positions one move from the end, so that winners occur
    rng = np.random.default_rng(3)
    n = len(q)
    ply = rng.integers(0, 400, n).astype(np.int32)
    gid = rng.integers(0, 2 ** 40, n).astype(np.int64)
    ref = eng.select_moves_host(q)
    want = np.zeros((n, 32), np.int8)
    want_win = np.zeros(n, np.int8)
    H.advance(ref["chosen"], want, 777, ply, gid, want_win)
    got = np.zeros((n, 32), np.int8)
    win = np.full(n, 9, np.int8)
    val = np.zeros(n, np.float32)
    nseq = np.zeros(n, np.int32)
    cuts = [0, 1, 7000, 7001, n]
    for lane, (lo, hi) in enumerate(zip(cuts[:-1], cuts[1:])):
        eng.play_ply_host_async(lane, q[lo:hi], ply[lo:hi], gid[lo:hi], got[lo:hi], win[lo:hi], val[lo:hi], nseq[lo:hi], dice_seed=777)
    for lane in range(4):
        eng.wait(lane)
    ok = ref["n_seq"] > 0

    def check():
        assert np.array_equal(got, want)
        assert np.array_equal(win, want_win) and (want_win >= 0).any()
        assert np.array_equal(nseq, ref["n_seq"])
        assert np.array_equal(val[ok].view(np.uint32), ref["value"][ok].view(np.uint32))
    check()
    # the same batches again on the same lanes: each launch now walks its queue in the order the previous call left
    # for its OUTPUTS (a poor order for these inputs) - results must not depend on it
    for rep in range(2):
        got[:] = 0; win[:] = 9; val[:] = 0; nseq[:] = 0
        for lane, (lo, hi) in enumerate(zip(cuts[:-1], cuts[1:])):
            eng.play_ply_host_async(lane, q[lo:hi], ply[lo:hi], gid[lo:hi], got[lo:hi], win[lo:hi], val[lo:hi], nseq[lo:hi], dice_seed=777)
        for lane in range(4):
            eng.wait(lane)
        check()
    # and a follow-up ply on the advanced records (the order left by the previous call is now the right one)
    live = want_win < 0
    q2 = np.ascontiguousarray(want[live][:7000])
    ref2 = eng.select_moves_host(q2)
    want2 = np.zeros_like(q2)
    H.advance(ref2["chosen"], want2, 777, ply[:7000] + 1, gid[:7000])
    got2 = np.zeros_like(q2)
    eng.play_ply_host_async(0, q2, ply[:7000] + 1, gid[:7000], got2, dice_seed=777)
    eng.wait(0)
    assert np.array_equal(got2, want2)


def test_play_ply_restart_is_the_resident_population(eng, golden):
    """bgx_play_ply_restart_host_async driven from the host for a few hundred plies = the device-resident population of
    bgx_selfplay_step after the same number of plies: records, ply numbers and game ids of every slot, bit for bit
    (restarts in place with id + stride, first mover id % 2, Philox dice of ply 0), and the winners it reported are the
    games the resident population finished."""
    from bgx import host as H
    from bgx.lib import FIRST_PARITY
    from bgx.synth import START_BOARD
    eng.set_weights(*golden_weights(golden("model.npz"), "trained"))
    n, stride, plies = 3000, 3000, 150                     # trained weights: ~77 plies per game, so most slots restart once or twice
    eng.selfplay_init(n, first_id=0, id_stride=stride, seed=SEED, first_mover=FIRST_PARITY, traj_cap=0)
    st = eng.selfplay_step(plies)
    want_rec, want_ply, want_gid = eng.selfplay_read()
    # the same games from the host: opening records with the dice of ply 0
    gid = np.arange(n, dtype=np.int64)
    ply = np.zeros(n, np.int32)
    fresh = np.zeros((n, 32), np.int8)
    fresh[:, :24] = START_BOARD
    fresh[:, 28] = (gid & 1) ^ 1                           # bgx_advance_host flips the mover and rolls ply 0
    bufs = [H.advance(fresh, fresh.copy(), SEED, ply, gid), np.zeros((n, 32), np.int8)]
    win = np.zeros(n, np.int8)
    finished = p1 = 0
    cuts = [0, 1000, 1001, n]
    for step in range(plies):
        a, b = bufs[step & 1], bufs[1 - (step & 1)]
        for lane, (lo, hi) in enumerate(zip(cuts[:-1], cuts[1:])):
            eng.play_ply_restart_host_async(lane, a[lo:hi], ply[lo:hi], gid[lo:hi], stride, b[lo:hi], win[lo:hi], first_mover=FIRST_PARITY, dice_seed=SEED)
        for lane in range(3):
            eng.wait(lane)
        finished += int((win >= 0).sum())
        p1 += int((win == 0).sum())
    got = bufs[plies & 1]
    assert np.array_equal(ply, want_ply) and np.array_equal(gid, want_gid)
    assert np.array_equal(got[:, :29], want_rec[:, :29])                     # position + mover (the resident slot keeps no dice)
    assert finished == st["games_finished"] and p1 == st["p1_wins"] and finished > n


def test_select_moves_golden_games(eng, orc, golden):
    """The reference's own greedy games (model.make_move on the reference engine), ply by ply."""
    g = golden("games.npz")
    gm = golden("model.npz")
    for name in g["names"]:
        name = str(name)
        tag = "rand" if name.startswith("rand") else "trained"
        w = golden_weights(gm, tag)
        eng.set_weights(*w)
        q = records_from(g[f"{name}.pre"], g[f"{name}.player"], g[f"{name}.dice"])
        out = eng.select_moves_host(q)
        assert np.array_equal(out["n_seq"], g[f"{name}.nseq"].astype(np.int32))
        same = (out["chosen"][:, :28] == g[f"{name}.after"]).all(1)
        for t in np.nonzero(~same)[0]:
            check_choice(orc, w, q[t], out["chosen"][t], out["value"][t], int(out["n_seq"][t]))
        exact_moves = (out["moves"].reshape(-1, 8) == g[f"{name}.chosen"].reshape(-1, 8)).all(1) & \
                      (out["moves_len"] == g[f"{name}.chosen_len"])
        # same afterstate, usually the reference's own sequence: torch's batched sgemm gives identical rows values that differ
        # in the last bit, so ITS arg-max may land on a later duplicate of the best afterstate; against the oracle (one value
        # per state) the sequences are identical on all 60,000 positions of test_select_moves_large_sample_vs_oracle
        assert exact_moves[same].mean() > 0.85
        assert same.mean() > (0.8 if tag == "rand" else 0.97), (name, same.mean())


def test_select_moves_epsilon_one_is_uniform_over_sequences(eng, orc, golden):
    """epsilon = 1: sequence floor(x1 * N / 2^32) of Philox(seed; 0, q, 0, 2), duplicates weighted (model.py:205-206)."""
    from bgx.synth import make_queries
    eng.set_weights(*golden_weights(golden("model.npz"), "rand"))
    q, _ = make_queries(800, seed=5)
    out = eng.select_moves_host(q, epsilon=1.0, seed=1234567)
    for i, r in enumerate(q):
        mv, ln, st = orc.turn_sequences(r[:28].astype(np.int32), r[28], r[29], r[30])
        assert out["n_seq"][i] == len(ln)
        if len(ln) == 0:
            continue
        x = orc.philox(1234567, 0, i, 0, 2)
        k = (x[1] * len(ln)) >> 32
        assert np.array_equal(out["chosen"][i, :28], st[k].astype(np.int8))
        assert out["moves_len"][i] == ln[k] and np.array_equal(out["moves"][i], mv[k])


# ------------------------------------------------------------------ self-play population

def verify_trajectory(orc, w, pre, cho, gid, first_rule_rolloff=True):
    """Step the oracle through an exported GPU trajectory (dice spec, legality, choice, turn order)."""
    T = len(pre)
    assert T > 0
    soft = 0
    if first_rule_rolloff:
        k = 0
        while True:
            x = orc.philox(SEED, k, gid, 0, 1)
            s1, s2 = orc.die(x[0]) + orc.die(x[1]), orc.die(x[2]) + orc.die(x[3])
            if s1 != s2:
                break
            k += 1
        assert pre[0, 28] == (0 if s1 > s2 else 1)
    from bgx.synth import START_BOARD
    assert np.array_equal(pre[0, :24], START_BOARD) and not pre[0, 24:28].any()
    for t in range(T):
        x = orc.philox(SEED, t, gid, 0, 0)
        assert (orc.die(x[0]), orc.die(x[1])) == (int(pre[t, 29]), int(pre[t, 30])), (gid, t)
        soft += check_choice(orc, w, pre[t], cho[t])
        if t + 1 < T:
            assert np.array_equal(pre[t + 1, :28], cho[t, :28]), (gid, t)     # next pre-move state = chosen afterstate
            assert pre[t + 1, 28] == 1 - pre[t, 28]                           # train.py:119-120
            assert orc.game_over(cho[t, :28].astype(np.int32)) == -1
    return soft


@pytest.mark.parametrize("tag", ["trained", "rand"])
def test_selfplay_round_trajectories(eng, orc, golden, tag):
    w = golden_weights(golden("model.npz"), tag)
    eng.set_weights(*w)
    n = 48
    eng.selfplay_init(n, first_id=1000, id_stride=n, seed=SEED, traj_cap=2048, record_chosen=True)
    st = eng.selfplay_round()
    rec, ply, gid = eng.selfplay_read()
    assert st["games_finished"] == n and st["truncated"] == 0
    assert st["plies"] == int(ply.sum())
    assert np.array_equal(gid, 1000 + np.arange(n))
    assert st["p1_wins"] == int((rec[:, 31] == 1).sum())
    for slot in range(0, n, 6):
        pre, cho = eng.export_trajectory(slot)
        assert len(pre) == ply[slot]
        verify_trajectory(orc, w, pre, cho, int(gid[slot]))
        winner = orc.game_over(cho[-1, :28].astype(np.int32))
        assert winner == int(rec[slot, 31]) - 1
        assert np.array_equal(rec[slot, :28], cho[-1, :28])
    # a second round continues with the next ids
    eng.selfplay_next_round()
    rec2, ply2, gid2 = eng.selfplay_read()
    assert np.array_equal(gid2, gid + n) and not ply2.any() and not rec2[:, 31].any()


def test_selfplay_golden_game_ids(eng, golden):
    """Same seed and game ids as the reference-played golden games: identical trajectories
    (trained weights: the value gaps are far above fp32 noise)."""
    g = golden("games.npz")
    eng.set_weights(*golden_weights(golden("model.npz"), "trained"))
    eng.selfplay_init(3, first_id=5, id_stride=3, seed=int(g["seed"]), traj_cap=1024, record_chosen=True)
    eng.selfplay_round()
    rec, ply, gid = eng.selfplay_read()
    for slot, name in enumerate(("trained5", "trained6", "trained7")):
        pre, cho = eng.export_trajectory(slot)
        gp = g[f"{name}.pre"]
        same = min(len(pre), len(gp))
        agree = (pre[:same, :29] == np.concatenate([gp, g[f"{name}.player"][:, None]], 1)[:same]).all(1)
        first_diff = same if agree.all() else int(np.argmin(agree))
        assert first_diff >= same - 1 or first_diff > 20, (name, first_diff)
        if agree.all() and len(pre) == len(gp):
            assert int(rec[slot, 31]) - 1 == int(g[f"{name}.winner"])
            assert np.array_equal(pre[:, 29:31], g[f"{name}.dice"])


def test_thousand_random_games_bit_exact(eng, orc, golden, request):
    """BASELINE.json configs[0] on the GPU: 1,000 random-vs-random games (epsilon = 1, the policy of
    benchmark.py:54-61 / model.py:205-206: uniform over the SEQUENCES, duplicates weighted) with the seeded
    Philox dice.  No floating point decides anything here, so every ply of every game must be bit-exact:
    dice, sequence count, the sequence the draw selects in reference order, the resulting 28-int state,
    turn order, game length and winner - against the oracle for all games and against the UNMODIFIED
    reference engine (oracle/_ref, when it was built) for a subset."""
    from bgx.synth import START_BOARD
    from oracle.oracle import RefHarness
    ref = RefHarness() if RefHarness.available() else None
    eng.set_weights(*golden_weights(golden("model.npz"), "rand"))
    n = 1000
    eng.selfplay_init(n, first_id=0, id_stride=n, seed=SEED, first_mover=1, traj_cap=2048, record_chosen=True)
    st = eng.selfplay_round(epsilon=1.0)
    rec, ply, gid = eng.selfplay_read()
    assert st["games_finished"] == n and st["truncated"] == 0 and st["plies"] == int(ply.sum())
    wins = 0
    for slot in range(n):
        g = int(gid[slot])
        pre, cho = eng.export_trajectory(slot)
        assert len(pre) == ply[slot] > 0
        s = np.zeros(28, np.int32)
        s[:24] = START_BOARD
        mover = g & 1                                                   # FIRST_PARITY: first mover = id % 2
        for t in range(len(pre)):
            x = orc.philox(SEED, t, g, 0, 0)
            d1, d2 = orc.die(x[0]), orc.die(x[1])
            assert np.array_equal(pre[t, :28], s.astype(np.int8)) and (int(pre[t, 28]), int(pre[t, 29]), int(pre[t, 30])) == (mover, d1, d2), (g, t)
            mv, ln, states = orc.turn_sequences(s, mover, d1, d2)
            if ref is not None and slot % 50 == 0:
                rmv, rln, rstates = ref.turn_sequences(s, mover, d1, d2)
                assert np.array_equal(mv, rmv) and np.array_equal(ln, rln) and np.array_equal(states, rstates), (g, t)
            if len(ln):
                e = orc.philox(SEED, t, g, 0, 2)
                assert np.float32(e[0]) * np.float32(2.3283064365386963e-10) < np.float32(1.0)   # the explore draw
                s = states[(e[1] * len(ln)) >> 32].astype(np.int32)
            assert np.array_equal(cho[t, :28], s.astype(np.int8)), (g, t)
            assert int(cho[t, 31]) == (1 if len(ln) and ln[(e[1] * len(ln)) >> 32] > 0 else 0), (g, t)
            over = orc.game_over(s)
            assert (over >= 0) == (t == len(pre) - 1), (g, t)
            mover ^= 1
        assert over == int(rec[slot, 31]) - 1
        wins += over == 0
    assert wins == st["p1_wins"]


def test_selfplay_step_restarts_and_rank_invariance(eng, golden):
    """Slots sharded over 'ranks' play the same games as one big population (ids = first_id + slot, stride = global)."""
    eng.set_weights(*golden_weights(golden("model.npz"), "trained"))
    G = 64
    eng.selfplay_init(G, first_id=0, id_stride=G, seed=SEED, first_mover=1)
    tot = {"plies": 0, "games_finished": 0}
    for _ in range(4):
        st = eng.selfplay_step(40)
        assert st["plies"] == G * 40
        for k in tot:
            tot[k] += st[k]
    full = eng.selfplay_read()
    assert tot["games_finished"] > 0 and (full[2] >= G).any()              # somebody restarted in place
    halves = []
    for r in range(2):
        eng.selfplay_init(G // 2, first_id=r * G // 2, id_stride=G, seed=SEED, first_mover=1)
        for _ in range(4):
            eng.selfplay_step(40)
        halves.append(eng.selfplay_read())
    for k in range(3):
        assert np.array_equal(full[k], np.concatenate([h[k] for h in halves]))


# ------------------------------------------------------------------ TD(lambda)

def td_game_bound(tag, k):
    """What a SINGLE game's max|dw - dw_ref| / max|dw_ref| may be: the worst of the 1,024 fixture games + 20 % (GPU_VS_TORCH below,
    all coordinates).  1e-5 holds for the median game, not for every game - for no fp32 implementation (RESTATEMENT_VS_TORCH)."""
    return 1.2 * GPU_VS_TORCH[tag]["all"][k][2]


def test_td_replay_host_golden(eng, golden):
    """apply_td_updates (train.py:124-172) on the reference's own trajectories (five reference-played games)."""
    g = golden("games.npz")
    gm = golden("model.npz")
    for name in g["names"]:
        name = str(name)
        tag = "rand" if name.startswith("rand") else "trained"
        w0 = golden_weights(gm, tag)
        eng.set_weights(*w0)
        rec = records_from(g[f"{name}.pre"], g[f"{name}.player"])
        new, sq = eng.td_replay_host(rec, int(g[f"{name}.winner"]) == 0, float(g[f"{name}.lr"]), float(g[f"{name}.lam"]))
        for a, b, k in zip(new, w0, ("W1", "b1", "w2", "b2")):
            ref_new = g[f"{name}.new_{k}"].reshape(-1)
            dref = ref_new.astype(np.float64) - np.asarray(b).reshape(-1)
            dgot = np.asarray(a).reshape(-1).astype(np.float64) - np.asarray(b).reshape(-1)
            assert np.max(np.abs(dgot - dref)) <= td_game_bound(tag, k) * np.max(np.abs(dref)), (name, k)
        assert np.max(np.abs(np.sqrt(sq) - np.sqrt(g[f"{name}.losses"]))) <= 1e-5, name


@pytest.mark.parametrize("tag", ["trained", "rand"])
def test_td_round_delta_is_sum_of_per_game_replays(eng, orc, golden, tag):
    import torch
    w0 = golden_weights(golden("model.npz"), tag)
    eng.set_weights(*w0)
    # 48 games: a TD error is the difference of two fp32 values near 0.5 (1e-4 apart with random-init weights),
    # so any two fp32 implementations differ by ~1e-5 of max|dw| on a dozen games (tools/td_err_probe.py:
    # oracle vs torch 5e-6, either GPU kernel vs oracle 0.5-1.5e-5); over 48 games the noise averages to ~2e-6
    n = 48
    eng.selfplay_init(n, first_id=1000, id_stride=n, seed=SEED, traj_cap=2048)
    eng.selfplay_round()
    rec, ply, gid = eng.selfplay_read()
    delta = torch.zeros(25604, device="cuda", dtype=torch.float32)
    st = eng.td_replay(0.1, 0.9, delta)
    torch.cuda.synchronize()
    assert st["td_steps"] == int(ply.sum()) and st["games_finished"] == n
    got = delta.cpu().numpy()
    flat0 = np.concatenate([np.asarray(a, np.float32).reshape(-1) for a in w0])
    want = np.zeros(25601, np.float64)
    sq_total = 0.0
    for slot in range(n):
        pre, _ = eng.export_trajectory(slot)
        X = np.concatenate([orc.encode(pre[t:t + 1, :28].astype(np.int32), int(pre[t, 28])) for t in range(len(pre))])
        new, sq = orc.td_replay(w0, X, rec[slot, 31] == 1, 0.1, 0.9)
        want += np.concatenate([np.asarray(a, np.float32).reshape(-1) for a in new]).astype(np.float64) - flat0
        sq_total += float(sq.sum())
    for lo, hi, k in ((0, 25344, "W1"), (25344, 25472, "b1"), (25472, 25600, "w2"), (25600, 25601, "b2")):
        tol = 1e-5 * np.max(np.abs(want[lo:hi])) + n * np.spacing(np.float32(np.max(np.abs(flat0[lo:hi]))))
        assert np.max(np.abs(got[lo:hi] - want[lo:hi])) <= tol, k
    assert not got[25601:].any()
    assert abs(st["td_sq_error"] - sq_total) <= 1e-4 * max(sq_total, 1e-12) + 1e-9
    # weights unchanged by the replay; apply_delta adds scale * delta
    assert np.array_equal(np.concatenate([np.asarray(a).reshape(-1) for a in eng.get_weights()]), flat0)
    eng.apply_delta(delta, 0.5)
    after = np.concatenate([np.asarray(a).reshape(-1) for a in eng.get_weights()])
    assert np.allclose(after, flat0 + 0.5 * got[:25601], rtol=0, atol=1e-7 * np.max(np.abs(flat0)) + 1e-9)


# max|dw - dw_ref| / max|dw_ref| per game of bgx_td_replay_host against the reference's own apply_td_updates (torch) on the
# 1,024 fixture trajectories per weight set, (p50, p99, max) as measured on a B200 (tools/td_parity_probe.py,
# profiles/r2_td_parity.json).  "fixture": over the 320 coordinates per game the committed fixture holds; "all": over all
# 25,601 coordinates against the live torch replay (tests/ref_td.py, which reproduces the fixture bit for bit on the box).
# The asserted bounds are these + 20 %.  For scale, the same distances for the fp32 C restatement of the reference are
# RESTATEMENT_VS_TORCH in tests/test_oracle_golden.py: no fp32 implementation sits within 1e-5 of torch on every game.
GPU_VS_TORCH = {
    "rand": {"fixture": {"W1": (3.42e-6, 1.21e-5, 1.70e-5), "b1": (3.08e-6, 1.39e-5, 2.32e-5), "w2": (1.06e-6, 3.99e-6, 7.07e-6), "b2": (8.09e-7, 3.67e-6, 6.80e-6)},
             "all": {"W1": (7.78e-6, 2.01e-5, 2.84e-5), "b1": (3.22e-6, 1.44e-5, 2.34e-5), "w2": (1.07e-6, 3.99e-6, 7.07e-6), "b2": (8.09e-7, 3.67e-6, 6.80e-6)}},
    "trained": {"fixture": {"W1": (9.25e-6, 4.33e-5, 8.39e-5), "b1": (5.13e-6, 3.74e-5, 7.02e-5), "w2": (3.06e-6, 1.25e-5, 2.29e-5), "b2": (4.71e-7, 2.94e-5, 1.87e-4)},
                "all": {"W1": (1.25e-5, 4.51e-5, 8.39e-5), "b1": (8.54e-6, 3.74e-5, 7.02e-5), "w2": (3.20e-6, 1.26e-5, 2.29e-5), "b2": (4.71e-7, 2.94e-5, 1.87e-4)}},
}


@pytest.mark.parametrize("tag", ["rand", "trained"])
def test_td_per_game_parity_vs_the_reference_update(eng, orc, golden, tag):
    """SURVEY 8d config 4: the per-game weight change of k_td_replay on 1,024 GPU-exported self-play trajectories per weight
    set against the REFERENCE'S OWN apply_td_updates (train.py:124-172, torch autograd) from the same snapshot:
      (i)   against the committed results of the unmodified reference (tests/golden/td_parity.npz) on every game;
      (ii)  against a live torch replay of all games over all 25,601 coordinates, after checking that this replay reproduces
            the fixture bit for bit (so (ii) is a statement about the reference, not about a restatement);
      (iii) against the exact float64 replay the kernel is as close as torch itself is;
      (iv)  the per-step TD errors agree at the value tolerance."""
    from oracle.oracle import td_replay_f64
    from ref_td import replay_many
    from td_fixture import BOUNDS, TENSORS, TdFixture, engine_errors, quantiles
    fx = TdFixture(golden, tag)
    err, worst_sq, news = engine_errors(eng, fx)
    assert worst_sq <= 1e-5                                                  # (iv)
    got = quantiles(err)
    for name in TENSORS:                                                     # (i)
        for g_, w_, what in zip(got[name], GPU_VS_TORCH[tag]["fixture"][name], ("p50", "p99", "max")):
            assert g_ <= 1.2 * w_, (tag, name, what, g_, w_)

    def enc(r):
        return np.concatenate([orc.encode(r[t:t + 1, :28].astype(np.int32), int(r[t, 28])) for t in range(len(r))])
    X = [enc(fx.trajectory(g)) for g in range(fx.n)]
    live = replay_many([(fx.w0, X[g], int(fx.p1_won[g]), fx.lr, fx.lam) for g in range(fx.n)])
    full = np.zeros((fx.n, 4))
    for g, (new, sq) in enumerate(live):                                     # (ii)
        assert np.array_equal(new[fx.coords(g)], fx.new_at[g]), ("the live torch replay is not the fixture's", tag, g)
        d_ref = new.astype(np.float64) - fx.w0_flat
        d = np.abs(news[g].astype(np.float64) - new.astype(np.float64))
        for k in range(4):
            full[g, k] = d[BOUNDS[k]:BOUNDS[k + 1]].max() / np.abs(d_ref[BOUNDS[k]:BOUNDS[k + 1]]).max()
    got = quantiles(full)
    for name in TENSORS:
        for g_, w_, what in zip(got[name], GPU_VS_TORCH[tag]["all"][name], ("p50", "p99", "max")):
            assert g_ <= 1.2 * w_, (tag, name, "all coordinates", what, g_, w_)
    games = range(0, fx.n, 4)                                                # (iii) 256 games, all coordinates
    e_gpu, e_ref = np.zeros((len(games), 4)), np.zeros((len(games), 4))
    for i, g in enumerate(games):
        new64 = np.concatenate([np.asarray(a).reshape(-1) for a in td_replay_f64(fx.w0, X[g], fx.p1_won[g], fx.lr, fx.lam)])
        d64 = new64 - fx.w0_flat
        for k in range(4):
            sl = slice(BOUNDS[k], BOUNDS[k + 1])
            e_gpu[i, k] = np.abs(news[g][sl] - new64[sl]).max() / np.abs(d64[sl]).max()
            e_ref[i, k] = np.abs(live[g][0][sl] - new64[sl]).max() / np.abs(d64[sl]).max()
    for k, name in enumerate(TENSORS):
        # measured kernel / torch: W1 0.98 / 0.98 / 1.11 (p50 / p99 / max), the small tensors 0.7 .. 1.23 (b2 is one number)
        for q, slack in ((0.5, 1.3), (0.99, 1.3), (1.0, 1.4)):
            assert np.quantile(e_gpu[:, k], q) <= slack * np.quantile(e_ref[:, k], q), (tag, name, q)


def test_td_replay_scheduled_follows_the_reference_schedule_per_game(eng, golden):
    """train.py:538 calls update_learning_params(games_done + k + 1) before the k-th game of a round (model.py:69-73).
    bgx_td_replay_scheduled looks that schedule up per game: across the 30,000-game boundary of lambda and the 40,000-game
    boundary of lr the summed weight change equals the sum of fixed-(lr, lambda) replays of the games on either side."""
    import torch
    from bgx.model import TDLGammonModel
    w0 = golden_weights(golden("model.npz"), "trained")
    eng.set_weights(*w0)
    n = 64
    eng.selfplay_init(n, first_id=0, id_stride=n, seed=SEED, traj_cap=2048)
    eng.selfplay_round()
    m = TDLGammonModel()
    delta = torch.zeros(25604, device="cuda", dtype=torch.float32)
    for boundary in (30000, 40000, 120000):
        games_done = boundary - 40                                          # slots 0..38 are episodes <= boundary - 1, the rest beyond
        eng.td_replay_scheduled(games_done, delta)
        got = delta.cpu().numpy().astype(np.float64)
        want = np.zeros(25604)
        trajs = [eng.export_trajectory(s)[0] for s in range(n)]
        rec, _, _ = eng.selfplay_read()
        flat0 = np.concatenate([np.asarray(a, np.float32).reshape(-1) for a in w0])
        params = set()
        for s in range(n):
            m.update_learning_params(games_done + s + 1)
            params.add((m.learning_rate, m.lambda_decay))
            new, _ = eng.td_replay_host(trajs[s], rec[s, 31] == 1, m.learning_rate, m.lambda_decay)
            want[:25601] += np.concatenate([np.asarray(a, np.float32).reshape(-1) for a in new]).astype(np.float64) - flat0
        assert len(params) == 2, (boundary, params)                          # the round really straddles a schedule step
        assert np.max(np.abs(got - want)) <= 2e-6 * np.max(np.abs(want)) + n * np.spacing(np.float32(np.max(np.abs(flat0))))
    eng.set_weights(*w0)


def test_gpu_trainer_owns_its_engine_and_checkpoints_see_its_weights(golden, tmp_path):
    """A GpuTrainer keeps the live weights in a private engine: batched calls through the module's own engine neither
    overwrite them nor free its population, and save_checkpoint writes the trained weights (ADVICE r1)."""
    import torch
    from bgx.model import TDLGammonModel
    from bgx.train import GpuTrainer, play_games_batch, save_checkpoint
    torch.manual_seed(3)
    m = TDLGammonModel()
    before = np.concatenate([a.reshape(-1) for a in m.weights_np()])
    tr = GpuTrainer(m, 64, delta_scale=1.0 / 64)
    try:
        tr.round()
        trained = np.concatenate([np.asarray(a).reshape(-1) for a in tr.eng.get_weights()])
        assert not np.array_equal(trained, before)
        games = play_games_batch(m, 4, seed=SEED)                            # the module's own engine: stale weights, own population
        assert len(games) == 4
        assert np.array_equal(np.concatenate([np.asarray(a).reshape(-1) for a in tr.eng.get_weights()]), trained)
        st = tr.round()                                                      # the trainer's population is intact
        assert st["games_finished"] == 64 and st["td_steps"] > 0
        trained = np.concatenate([np.asarray(a).reshape(-1) for a in tr.eng.get_weights()])
        path = str(tmp_path / "ckpt.pth")
        save_checkpoint(m, path)                                             # pulls the trainer's weights first
        sd = torch.load(path, map_location="cpu", weights_only=True)
        saved = np.concatenate([sd[k].numpy().reshape(-1) for k in ("fc1.weight", "fc1.bias", "fc2.weight", "fc2.bias")])
        assert np.array_equal(saved, trained)
        # the module's engine is refreshed only when the module's parameters changed
        e = m.engine(0)
        assert np.array_equal(np.concatenate([np.asarray(a).reshape(-1) for a in e.get_weights()]), trained)
    finally:
        tr.eng.close()


# ------------------------------------------------------------------ batched head-to-head (train.py:262-302, benchmark.py:64-130)

def test_arena_games_replay_through_the_oracle(orc, golden):
    """Every ply of every head-to-head game: dice follow the Philox rule, the mover alternates, the policy that
    owns the mover picked the oracle's move (within the value tolerance), the winner is the reference's."""
    from bgx.evaluate import Arena
    gm = golden("model.npz")
    wa, wb = golden_weights(gm, "trained"), golden_weights(gm, "rand")
    n = 24
    side = (np.arange(n) % 2).astype(np.int8)
    first = ((np.arange(n) // 2) % 2).astype(np.int8)
    arena = Arena(0)
    try:
        res = arena.play(wa, wb, side, first, seed=SEED, record=True)
    finally:
        arena.close()
    assert (res["winner"] >= 0).all()
    state = {i: None for i in range(n)}
    count = np.zeros(n, np.int64)
    soft = 0
    for ply, idx, q, ch in res["log"]:
        for j, g in enumerate(idx):
            r = q[j]
            x = orc.philox(SEED, ply, int(g))
            assert (int(r[29]), int(r[30])) == (orc.die(x[0]), orc.die(x[1]))
            assert int(r[28]) == (int(first[g]) ^ (ply & 1))
            if state[g] is None:
                assert np.array_equal(r[:24], START_BOARD_NP) and not r[24:28].any()
            else:
                assert np.array_equal(r[:28], state[g])
            w = wa if int(r[28]) == int(side[g]) else wb
            soft += check_choice(orc, w, r, ch[j])
            state[g] = ch[j, :28].copy()
            count[g] += 1
    assert soft <= 0.1 * count.sum()
    for g in range(n):
        assert orc.game_over(state[g].astype(np.int32)) == int(res["winner"][g])
        assert count[g] == res["plies"][g]


def test_arena_reference_evaluation_loops(golden):
    """evaluate_parallel / play_vs_random / play_vs_model on the GPU: a trained net beats the random policy and the
    random-init net; a net against itself is even; results are reproducible."""
    from bgx.evaluate import Arena, evaluate, play_vs_model, play_vs_random
    gm = golden("model.npz")
    wt, wr = golden_weights(gm, "trained"), golden_weights(gm, "rand")
    arena = Arena(0)
    try:
        rate, avg_len = play_vs_random(arena, wt, 512)
        assert rate > 0.9 and 20 < avg_len < 200
        assert play_vs_random(arena, wt, 512) == (rate, avg_len)          # random draws are seeded too
        assert evaluate(arena, wt, wr, 512) > 0.85
        r1, _ = play_vs_model(arena, wt, wt, 2048)
        assert 0.42 < r1 < 0.58
    finally:
        arena.close()


def test_play_games_batch_feeds_the_reference_td_update(eng, golden):
    """bgx.train.play_games_batch returns play_game's tuples; the reference-contract apply_td_updates (torch autograd,
    CPU) on those states and the GPU replay of the same trajectory give the same weights."""
    import torch
    from bgx.model import TDLGammonModel
    from bgx.train import play_games_batch
    from ref_td import apply_td_updates
    W1, b1, w2, b2 = golden_weights(golden("model.npz"), "trained")
    sd = {"fc1.weight": torch.from_numpy(W1), "fc1.bias": torch.from_numpy(b1),
          "fc2.weight": torch.from_numpy(w2), "fc2.bias": torch.from_numpy(b2)}
    m = TDLGammonModel()
    m.load_state_dict(sd)
    games = play_games_batch(m, 6, seed=SEED, first_id=40)
    assert len(games) == 6
    for winner, states, total in games:
        assert winner in (0, 1) and len(states) == total + 1
        assert states[0].shape == (198,) and states[0].dtype == np.float32
        assert states[0][:192].sum() == 26.0 and states[0][192] + states[0][193] == 1.0      # the opening position
    winner, states, _ = min(games, key=lambda g: len(g[1]))
    m.update_learning_params(1)
    m.initialize_traces()
    apply_td_updates(m, torch.optim.SGD(m.parameters(), lr=0.1), states, winner == 0)
    eng.set_weights(W1, b1, w2, b2)
    # the same trajectory as records: slot order is game order
    idx = [i for i, g in enumerate(games) if g[1] is states][0]
    pre, _ = m.engine(0).export_trajectory(idx)
    new, _ = eng.td_replay_host(pre, winner == 0, m.learning_rate, m.lambda_decay)
    for a, name in zip(new, ("fc1.weight", "fc1.bias", "fc2.weight", "fc2.bias")):
        ref = m.state_dict()[name].numpy().reshape(-1)
        d_ref = ref - sd[name].numpy().reshape(-1)
        k = {"fc1.weight": "W1", "fc1.bias": "b1", "fc2.weight": "w2", "fc2.bias": "b2"}[name]
        assert np.max(np.abs(np.asarray(a).reshape(-1) - ref)) <= td_game_bound("trained", k) * np.max(np.abs(d_ref)), name


# ------------------------------------------------------------------ the pybind11 module's batched entry points

def test_pybind_batch_engine_matches_the_c_abi(eng, golden):
    """backgammon_env.BatchEngine (the batched entry points the reference's binding file gains, backgammon_bindings.cpp
    + INTEGRATION.md) gives what the ctypes mirror of the same C-ABI gives: enumeration, make_moves, one loop iteration of
    play_game, a self-play round with exported trajectories, and the TD(lambda) round."""
    import bgx  # noqa: F401  (puts the in-tree module directory on sys.path)
    import backgammon_env as bg
    from bgx import host as H
    from bgx.synth import make_queries
    w = golden_weights(golden("model.npz"), "trained")
    eng.set_weights(*w)
    be = bg.BatchEngine(0)
    be.set_weights(*w)
    for a, b in zip(be.get_weights(), w):
        assert np.array_equal(np.asarray(a).reshape(-1), np.asarray(b).reshape(-1))
    q, _ = make_queries(3000, seed=2024)
    off, mv, ln, st = be.evaluate_turn_sequences(q)
    off2, mv2, ln2, st2 = eng.enumerate_host(q)
    assert np.array_equal(off, off2) and np.array_equal(mv, mv2) and np.array_equal(ln, ln2) and np.array_equal(st, st2)
    mm = be.make_moves(q)
    ref = eng.select_moves_host(q)
    for k in ("chosen", "moves", "moves_len", "n_seq"):
        assert np.array_equal(mm[k], ref[k]), k
    ply = np.arange(len(q), dtype=np.int32) % 300
    gid = np.arange(len(q), dtype=np.int64) * 7
    nxt, win, val, nseq = be.play_ply(q, ply, gid, dice_seed=99)
    want = np.zeros_like(nxt)
    want_win = np.zeros(len(q), np.int8)
    H.advance(ref["chosen"], want, 99, ply, gid, want_win)
    assert np.array_equal(nxt, want) and np.array_equal(win, want_win) and np.array_equal(nseq, ref["n_seq"])
    # a round of 32 games and its TD(lambda) update, on both front ends
    n = 32
    be.selfplay_init(n, first_id=500, id_stride=n, seed=SEED, traj_cap=1024, record_chosen=True)
    eng.selfplay_init(n, first_id=500, id_stride=n, seed=SEED, traj_cap=1024, record_chosen=True)
    s1, s2 = be.selfplay_round(), eng.selfplay_round()
    for k in ("plies", "sequences", "games_finished", "p1_wins", "truncated"):
        assert s1[k] == s2[k], k
    assert s1["games_finished"] == n
    r1, r2 = be.selfplay_read(), eng.selfplay_read()
    for a, b in zip(r1, r2):
        assert np.array_equal(a, b)
    for slot in (0, 13, 31):
        p1, c1 = be.export_trajectory(slot)
        p2, c2 = eng.export_trajectory(slot)
        assert np.array_equal(p1, p2) and np.array_equal(c1, c2)
    import torch
    delta_dev = torch.zeros(25604, dtype=torch.float32, device="cuda")
    t2 = eng.td_replay(0.1, 0.9, delta_dev)
    delta, t1 = be.td_round(0.1, 0.9, 1.0 / n)
    assert t1["td_steps"] == t2["td_steps"] == int(r1[1].sum())
    assert np.array_equal(delta, delta_dev.cpu().numpy()[:25601])
    eng.apply_delta(delta_dev, 1.0 / n)
    for a, b in zip(be.get_weights(), eng.get_weights()):
        assert np.array_equal(np.asarray(a).reshape(-1), np.asarray(b).reshape(-1))
    be.selfplay_next_round()
    assert not be.selfplay_read()[1].any()


# ------------------------------------------------------------------ the whole training loop, end to end

def test_gpu_trainer_learns_to_beat_the_random_policy():
    """BASELINE configs[3] as a function, not only as a throughput: rounds of self-play from one snapshot + exact TD(lambda)
    replay + mean of the per-game weight changes (bgx.train.GpuTrainer), from the reference's random initialisation
    (model.py:55-61), turn a net that is even with the random policy into one that beats it - a few seconds on a B200."""
    import torch
    from bgx.evaluate import Arena, play_vs_random
    from bgx.model import TDLGammonModel
    from bgx.train import GpuTrainer
    torch.manual_seed(0)
    m = TDLGammonModel()
    arena = Arena(0)
    try:
        before, _ = play_vs_random(arena, m.weights_np(), 1024)
        tr = GpuTrainer(m, 256, delta_scale=2.0 / 256)
        for _ in range(2000):
            st = tr.round(epsilon=0.0)
        tr.sync_model()
        after, avg_len = play_vs_random(arena, m.weights_np(), 1024)
    finally:
        arena.close()
    assert st["games_finished"] == 256 and st["truncated"] == 0
    assert before < 0.7 and after > 0.95, (before, after)
    assert avg_len < 90                               # it learnt to race: random-init games last ~109 plies
