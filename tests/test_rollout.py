"""Rollouts (DESIGN 7d, bgx_rollout): the dice rule, the outcome classes and the oracle restatement on the CPU; on the GPU the fused
rollout kernel against the host-driven loop over the one-ply kernel (bit for bit), against the CPU oracle under exact tie nets,
against two-ply's expectation at T = 1, as a pure function of its inputs, on its edge cases, against self-play statistics and
through every surface."""
import math

import numpy as np
import pytest
from conftest import golden_weights
from rollout_ref import MAX_PLIES, STREAM, dice, die_np, engine_ply, oracle_ply, outcome_class, philox_np, reduce_trials, rollout
from test_ply_exactness import integer_rule, tie_net

SEED = 0x5EED2026
START = np.array([2, 0, 0, 0, 0, -5, 0, -3, 0, 0, 0, 5, -5, 0, 0, 0, 3, 0, 5, 0, 0, 0, 0, -2], np.int8)
OUT_KEYS = ("mean", "std_err", "counts", "trial_value", "trial_outcome", "trial_plies")


def rec_of(board, bar=(0, 0), off=(0, 0), player=0):
    r = np.zeros(32, np.int8)
    r[:24] = board
    r[24:26] = bar
    r[26:28] = off
    r[28] = player
    return r


def positions(n, seed):
    from bgx.synth import make_queries
    q = make_queries(n, seed=seed)[0].copy()
    q[:, 29:] = 0                        # the dice of a query are ignored
    return q


def same(a, b, keys=OUT_KEYS, what=""):
    for k in keys:
        x, y = np.asarray(a[k]), np.asarray(b[k])
        assert x.shape == y.shape, (what, k, x.shape, y.shape)
        if x.dtype.kind == "f":
            assert np.array_equal(x.view(np.uint8), y.view(np.uint8)), (what, k)      # bit for bit, NaN included
        else:
            assert np.array_equal(x, y), (what, k)


# ------------------------------------------------------------------ CPU

def test_dice_rule(orc):
    """Philox stream 4, counter (k, t lo, t hi, 4), as the oracle's Philox and die; stratified ply 0 rolls t mod 36."""
    ts = np.array([0, 1, 35, 36, 1295, 2 ** 20 + 7, 2 ** 32 + 5, 2 ** 40 + 123], np.int64)
    for k in (0, 1, 2, 31, 32, 33, 4095):
        x = philox_np(SEED, np.full(len(ts), k), ts & 0xFFFFFFFF, ts >> 32, np.full(len(ts), STREAM))
        d1, d2 = dice(SEED, ts, k, stratify=False)
        for j, t in enumerate(ts):
            want = orc.philox(SEED, k, int(t) & 0xFFFFFFFF, int(t) >> 32, STREAM)
            assert [int(x[i][j]) for i in range(4)] == want
            assert (d1[j], d2[j]) == (orc.die(want[0]), orc.die(want[1]))
        if k > 0:                                                    # stratification touches ply 0 only
            s1, s2 = dice(SEED, ts, k, stratify=True)
            assert np.array_equal(s1, d1) and np.array_equal(s2, d2)
    # a stream of its own: not self-play's stream 0 on the same counters
    t = np.arange(4096, dtype=np.int64)
    a = philox_np(SEED, np.zeros(4096), t, 0, np.full(4096, STREAM))
    b = philox_np(SEED, np.zeros(4096), t, 0, np.zeros(4096))
    assert (a[0] != b[0]).mean() > 0.99
    # stratified ply 0: every ordered roll exactly trials / 36 times, in the order r = t mod 36
    for trials in (36, 72, 1296):
        d1, d2 = dice(SEED, np.arange(trials), 0, stratify=True)
        r = (d1.astype(int) - 1) * 6 + (d2.astype(int) - 1)
        assert np.array_equal(r, np.arange(trials) % 36)
        assert np.array_equal(np.bincount(r, minlength=36), np.full(36, trials // 36))
    # unstratified ply 0 is Philox like every other ply, and uniform
    d1, d2 = dice(SEED, np.arange(36 * 4000), 0, stratify=False)
    c = np.bincount((d1.astype(int) - 1) * 6 + d2 - 1, minlength=36)
    assert abs(c - 4000).max() < 5 * math.sqrt(4000)
    assert np.array_equal(die_np(np.array([0, 2 ** 32 - 1], np.uint64)), [1, 6])


def board(**points):
    """board(p19=2, ...) by point number (1..24); + PLAYER1, - PLAYER2"""
    b = np.zeros(24, np.int8)
    for k, v in points.items():
        b[int(k[1:]) - 1] = v
    return b


def test_home_boards_by_the_oracles_legal_moves(orc):
    """PLAYER1 bears off from board indices 18..23 (past point 24), PLAYER2 from 0..5: the direction outcome_class relies on."""
    def can_bear_off(s, player):
        return any(d == (25 if player == 0 else 0) for die in range(1, 7) for _, d in orc.legal_moves(s, player, die))

    for player, home, outside in ((0, range(18, 24), 17), (1, range(0, 6), 6)):
        sign = 1 if player == 0 else -1
        s = np.zeros(28, np.int32)
        for j, i in enumerate(home):
            s[i] = sign * (3 if j < 3 else 2)
        assert s[:24].sum() == sign * 15 and can_bear_off(s, player)
        s[home[0]] -= sign
        s[outside] = sign                                            # one checker just outside that home board
        assert not can_bear_off(s, player)


def test_outcome_classes():
    """Both winners, all three classes, each backgammon cause, from hand-built final boards."""
    cases = [
        # PLAYER1 won: PLAYER2 bore off 3 / nothing, far from PLAYER1's home / nothing, on the bar / nothing, in 19..24
        (rec_of(board(p1=-12), off=(15, 3)), 1),
        (rec_of(board(p1=-10, p18=-5), off=(15, 0)), 2),
        (rec_of(board(p1=-14), bar=(0, 1), off=(15, 0)), 3),
        (rec_of(board(p1=-14, p19=-1), off=(15, 0)), 3),
        (rec_of(board(p1=-14, p24=-1), off=(15, 0)), 3),
        # PLAYER2 won: the mirror image
        (rec_of(board(p24=12), off=(3, 15)), 4),
        (rec_of(board(p24=10, p7=5), off=(0, 15)), 5),
        (rec_of(board(p24=14), bar=(1, 0), off=(0, 15)), 6),
        (rec_of(board(p24=14, p6=1), off=(0, 15)), 6),
        (rec_of(board(p24=14, p1=1), off=(0, 15)), 6),
        # a backgammon needs a gammon first
        (rec_of(board(p1=-13), bar=(0, 1), off=(15, 1)), 1),
        (rec_of(board(p24=13, p1=1), off=(1, 15)), 4),
        # not over
        (rec_of(START), 0),
    ]
    for r, want in cases:
        assert outcome_class(r[:28]) == want, (r, want)


@pytest.mark.parametrize("kind", ("off", "bar"))
def test_oracle_restatement_under_tie_nets(orc, kind):
    """Under an exact tie net the restatement's every ply is the integer rule (the first sequence maximising the mover's
    feature), and a truncated trial's x_t is the oracle's fp32 value of the afterstate it chose."""
    w = tie_net(kind)
    ply, value = oracle_ply(orc, w)
    seen = []

    def on_ply(q, after, val, anyseq):
        seen.append((q.copy(), after.copy(), np.asarray(val).copy(), anyseq.copy()))

    pos = positions(4, seed=4242)
    out = rollout(ply, value, pos, 36, max_plies=0, on_ply=on_ply)
    assert (out["trial_outcome"] > 0).all()
    n_ply = 0
    for q, after, val, anyseq in seen[:40]:
        rule = integer_rule(orc, q, (kind,))
        has = rule["n_seq"] > 0
        assert np.array_equal(has, anyseq)
        assert np.array_equal(after[has], rule[kind]["after"][has])
        n_ply += len(q)
    assert n_ply > 1000
    cut = rollout(ply, value, pos, 36, max_plies=7)
    assert (cut["trial_plies"] <= 7).all() and (cut["trial_outcome"] == 0).any()
    last = seen[6]
    for t in (0, 1):
        m = (last[0][:, 28] == t) & last[3]
        if m.any():
            want = orc.forward(w, orc.encode(last[1][m].astype(np.int32), t))
            assert np.array_equal(np.asarray(last[2])[m].view(np.uint32), want.view(np.uint32))


# ------------------------------------------------------------------ GPU

@pytest.fixture(scope="module")
def eng():
    from bgx.engine import BatchEngine
    e = BatchEngine(0)
    yield e
    e.close()


def weights_of(golden, net):
    if net in ("trained", "rand"):
        return golden_weights(golden("model.npz"), net)
    return tie_net(net)


@pytest.mark.gpu
@pytest.mark.parametrize("net", ("trained", "rand"))
def test_rollout_is_the_host_driven_loop(eng, golden, net):
    """256 positions x 72 trials, T in {0, 1, 2, 7}, stratified and not: every per-trial value, outcome and ply count equals the
    host-driven loop over select_moves_host / evaluate_host, and every output equals the restatement's reduction bit for bit."""
    eng.set_weights(*weights_of(golden, net))
    pos = positions(256, seed=31337)
    ply, value = engine_ply(eng)
    for T in (0, 1, 2, 7):
        for strat in (True, False):
            got = eng.rollout_host(pos, 72, max_plies=T, seed=SEED, stratify=strat, per_trial=True)
            want = rollout(ply, value, pos, 72, max_plies=T, seed=SEED, stratify=strat)
            same(got, want, what=(net, T, strat))
            if T == 0:
                assert (got["trial_outcome"] > 0).all() and (got["counts"][:, 6] == 0).all()
            else:
                assert (got["trial_plies"] <= T).all()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ("off", "bar"))
def test_rollout_tie_nets_are_the_oracle(eng, orc, kind):
    """Under an exact tie net every ply of the kernel is the oracle's (the pick is an integer fact, no near-ties): 32 positions x 72
    trials, full games under `off`; under `bar`, whose games run to thousands of plies (the oracle scores every afterstate densely),
    cut at 48 plies.  Outcomes, ply counts and counts are equal, and so is x_t of every finished trial.  A truncated trial's x_t is a
    sigmoid, which the oracle takes from expf and the kernel from the SFU: equal to 2e-6 relative; the kernel's mean and std_err are
    the spec's reduction of its own per-trial values, bit for bit."""
    w = tie_net(kind)
    eng.set_weights(*w)
    pos = positions(32, seed=777)
    for T, strat in ((0 if kind == "off" else 48, True), (7, False)):
        got = eng.rollout_host(pos, 72, max_plies=T, seed=SEED, stratify=strat, per_trial=True)
        want = rollout(*oracle_ply(orc, w), pos, 72, max_plies=T, seed=SEED, stratify=strat)
        same(got, want, keys=("trial_outcome", "trial_plies", "counts"), what=(kind, T))
        fin = want["trial_outcome"] > 0
        assert np.array_equal(got["trial_value"][fin], want["trial_value"][fin])
        assert np.allclose(got["trial_value"][~fin], want["trial_value"][~fin], rtol=2e-6, atol=0)
        assert fin.any() and (T == 0 or (~fin).any())
        for i in range(len(pos)):
            m, se, _ = reduce_trials(got["trial_value"][i], got["trial_outcome"][i], got["trial_plies"][i])
            assert got["mean"][i] == m and np.array_equal(np.float64(got["std_err"][i]), np.float64(se))


@pytest.mark.gpu
def test_one_ply_rollout_is_twoply_expectation(eng, golden):
    """Roll out two-ply's pick A with the opponent on roll, T = 1, 36 stratified trials: float32(mean) is two-ply's E2(A) bit for
    bit wherever both float64 sums are exact (no reply can win: the opponent has <= 10 borne off; every x_t >= 2^-24)."""
    from bgx.synth import make_queries
    eng.set_weights(*golden_weights(golden("model.npz"), "trained"))
    q = make_queries(512, seed=2468)[0]
    two = eng.select_moves_2ply_host(q, max_candidates=0)
    A = two["chosen"].copy()
    p = q[:, 28].astype(np.int64)
    usable = (two["n_candidates"] > 0) & (A[:, 26] != 15) & (A[:, 27] != 15)
    A[:, 28] = 1 - p
    A[:, 29:] = 0
    A = A[usable]
    ro = eng.rollout_host(A, 36, max_plies=1, seed=SEED, stratify=True, per_trial=True)
    exact = (A[np.arange(len(A)), 26 + A[:, 28].astype(np.int64)] <= 10) & (ro["trial_value"] >= 2.0 ** -24).all(axis=1)
    assert exact.mean() > 0.9 and exact.sum() > 300
    v2 = two["value"][usable][exact]
    assert np.array_equal(ro["mean"][exact].astype(np.float32).view(np.uint32), v2.view(np.uint32))
    assert (ro["trial_plies"] == 1).all()


@pytest.mark.gpu
def test_rollout_is_a_pure_function(eng, golden):
    """The same positions give bit-identical outputs alone, inside a larger batch permuted and duplicated, under every chunking and
    every warps-per-CTA setting."""
    eng.set_weights(*golden_weights(golden("model.npz"), "trained"))
    pos = positions(24, seed=99)
    base = eng.rollout_host(pos, 72, seed=SEED, per_trial=True)
    other = positions(40, seed=100)
    big = np.concatenate([pos, other, pos[:8]])
    perm = np.random.default_rng(5).permutation(len(big))
    got = eng.rollout_host(big[perm], 72, seed=SEED, per_trial=True)
    inv = np.argsort(perm)
    where = inv[:24]
    same({k: v[where] for k, v in got.items()}, base, what="batch")
    dup = inv[64:72]
    same({k: v[dup] for k, v in got.items()}, {k: v[:8] for k, v in base.items()}, what="duplicates")
    for chunk in (72, 7 * 72, 0):
        eng.set_option("rollout_chunk", chunk)
        same(eng.rollout_host(pos, 72, seed=SEED, per_trial=True), base, what=("chunk", chunk))
    eng.set_option("rollout_chunk", 0)
    for warps in (16, 24, 32, 20):
        eng.set_option("rollout_warps", warps)
        same(eng.rollout_host(pos, 72, seed=SEED, per_trial=True), base, what=("warps", warps))
    # without the per-trial arrays: the same outputs (per-trial results in engine scratch)
    same(eng.rollout_host(pos, 72, seed=SEED), base, keys=("mean", "std_err", "counts"), what="scratch")


@pytest.mark.gpu
def test_rollout_edges(eng, golden):
    from bgx import lib as L
    eng.set_weights(*golden_weights(golden("model.npz"), "trained"))
    # finished positions: 0 plies, the exact outcome, std_err 0
    done = np.stack([rec_of(board(p1=-14, p19=-1), off=(15, 0), player=1), rec_of(board(p24=12), off=(3, 15), player=0)])
    o = eng.rollout_host(done, 36, seed=SEED, per_trial=True)
    assert (o["trial_plies"] == 0).all() and list(o["mean"]) == [1.0, 0.0] and list(o["std_err"]) == [0.0, 0.0]
    assert list(o["counts"][0]) == [0, 0, 36, 0, 0, 0, 0, 0] and list(o["counts"][1]) == [0, 0, 0, 36, 0, 0, 0, 0]
    # one trial: NaN standard error
    o = eng.rollout_host(positions(4, seed=1), 1, seed=SEED, stratify=False)
    assert np.isnan(o["std_err"]).all() and np.isfinite(o["mean"]).all()
    # the mover is blocked at ply 0 (PLAYER2 on the bar against a closed board): the trials still match the host loop
    closed = board(p19=2, p20=2, p21=2, p22=2, p23=2, p24=2, p11=3, p1=-4, p2=-4, p3=-3, p4=-3)
    blocked = np.stack([rec_of(closed, bar=(0, 1), player=1)] * 2)
    for T in (1, 0):
        got = eng.rollout_host(blocked, 36, max_plies=T, seed=SEED, per_trial=True)
        same(got, rollout(*engine_ply(eng), blocked, 36, max_plies=T, seed=SEED), what=("blocked", T))
    v = eng.evaluate_host(blocked[:1])[0]
    assert (got["trial_plies"] > 1).all()
    assert (eng.rollout_host(blocked, 36, max_plies=1, per_trial=True)["trial_value"] == v).all()
    # no positions
    o = eng.rollout_host(np.zeros((0, 32), np.int8), 36, per_trial=True)
    assert o["mean"].shape == (0,) and o["counts"].shape == (0, 8) and o["trial_value"].shape == (0, 36)
    # invalid arguments
    pos = positions(2, seed=3)
    for kw in ({"trials": 0}, {"trials": -36}, {"trials": 35}, {"trials": 72, "max_plies": MAX_PLIES + 1},
               {"trials": 72, "max_plies": -1}):
        with pytest.raises(L.BgxError) as ei:
            eng.rollout_host(pos, **kw)
        assert ei.value.code == L.E_INVALID
    assert eng.rollout_host(pos, 35, stratify=False)["mean"].shape == (2,)
    assert eng.rollout_host(pos, 36, max_plies=MAX_PLIES)["mean"].shape == (2,)
    rc = eng._lib.bgx_rollout_host(eng._h, pos.ctypes.data, 2, 36, 0, SEED, 2, None, None, None, None, None, None)
    assert rc == L.E_INVALID


@pytest.mark.gpu
def test_long_trials_under_the_bar_net(eng):
    """Under the bar net both sides hit whenever they can: trials of hundreds to thousands of plies, so each warp's 8-bit cache
    generation wraps inside a trial.  Still the host-driven loop bit for bit."""
    eng.set_weights(*tie_net("bar"))
    pos = positions(6, seed=4242)[4:]
    got = eng.rollout_host(pos, 36, max_plies=0, seed=SEED, per_trial=True)
    want = rollout(*engine_ply(eng), pos, 36, max_plies=0, seed=SEED)
    same(got, want, what="bar")
    assert np.median(got["trial_plies"]) > 300


@pytest.mark.gpu
def test_rollout_of_the_opening_agrees_with_selfplay(eng, golden):
    """2^16 unstratified trials of the opening, each player on roll, against P1's win and gammon fractions over 2^16 self-play
    games with the same first mover (an independent path: k_selfplay, other dice): within 4 sigma."""
    from bgx import lib as L
    eng.set_weights(*golden_weights(golden("model.npz"), "trained"))
    n = 1 << 16
    opening = np.stack([rec_of(START, player=0), rec_of(START, player=1)])
    ro = eng.rollout_host(opening, n, seed=SEED, stratify=False)
    assert (ro["counts"][:, 6] == 0).all()
    eng.selfplay_init(2 * n, seed=12345, first_mover=L.FIRST_PARITY)
    eng.selfplay_round()
    rec, ply, gid = eng.selfplay_read()
    first = gid % 2                                                  # BGX_FIRST_PARITY: game id % 2 moves first
    assert (rec[:, 31] > 0).all()
    for mover in (0, 1):
        m = first == mover
        games = rec[m]
        sp_win = (games[:, 31] == 1).mean()
        sp_gam = ((games[:, 31] == 1) & (games[:, 27] == 0)).mean()
        r_win = ro["counts"][mover, :3].sum() / n
        r_gam = ro["counts"][mover, 1:3].sum() / n
        assert r_win == ro["mean"][mover]
        for a, b in ((r_win, sp_win), (r_gam, sp_gam)):
            sigma = math.sqrt(a * (1 - a) / n + b * (1 - b) / m.sum())
            assert abs(a - b) < 4 * sigma, (mover, a, b, sigma)


@pytest.mark.gpu
def test_rollout_surfaces_agree(eng, golden):
    """ctypes host and device forms, the pybind module and TDLGammonModel.rollout_batch give the same results bit for bit."""
    import torch
    import backgammon_env as bg
    from bgx.model import TDLGammonModel
    w = golden_weights(golden("model.npz"), "trained")
    eng.set_weights(*w)
    pos = positions(16, seed=55)
    host = eng.rollout_host(pos, 72, max_plies=0, seed=SEED, per_trial=True)
    dev = eng.rollout(torch.from_numpy(pos).cuda(), 72, max_plies=0, seed=SEED, per_trial=True)
    torch.cuda.synchronize()
    same(host, {k: v.cpu().numpy() for k, v in dev.items()}, what="device")
    pb = bg.BatchEngine(0)
    pb.set_weights(*w)
    same(host, pb.rollout(pos, 72, 0, SEED, True, True), what="pybind")
    m = TDLGammonModel()
    W1, b1, w2, b2 = w
    m.load_state_dict({"fc1.weight": torch.from_numpy(W1), "fc1.bias": torch.from_numpy(b1),
                       "fc2.weight": torch.from_numpy(w2), "fc2.bias": torch.from_numpy(b2)})
    free = pos[(pos[:, 24] == 0) & (pos[:, 25] == 0)]               # the compat Game has no setter for the bar
    assert len(free) >= 4
    games = []
    for r in free:
        g = bg.Game(0)
        g.setGameBoard([int(x) for x in r[:24]])
        g.setBorneOffPieces(0, int(r[26]))
        g.setBorneOffPieces(1, int(r[27]))
        g.setTurn(int(r[28]))
        g.roll_dice()                                                # dice are ignored
        games.append(g)
    want = eng.rollout_host(free, 72, seed=SEED)
    rb = m.rollout_batch(games, trials=72, seed=SEED)
    assert np.array_equal(rb["p1_win"], want["mean"]) and np.array_equal(rb["std_err"], want["std_err"])
    assert np.array_equal(rb["outcomes"], want["counts"][:, :6] / 72.0)
    assert [list(g.getGameBoard()) for g in games] == [[int(x) for x in r[:24]] for r in free]
