"""Two-ply move selection (DESIGN 7c, bgx_select_moves_2ply): the CPU restatement against a direct torch restatement of the
spec, and the GPU path against the CPU restatement, against the one-ply kernel (K = 1), on its edge cases, as a pure function of
the query, through every surface, in head-to-head play."""
import numpy as np
import pytest
from conftest import golden_weights
from twoply_ref import ROLLS, WEIGHTS, twoply_batch

SEED = 0x5EED2026
START = np.array([2, 0, 0, 0, 0, -5, 0, -3, 0, 0, 0, 5, -5, 0, 0, 0, 3, 0, 5, 0, 0, 0, 0, -2], np.int8)


def rec_of(board, bar=(0, 0), off=(0, 0), player=0, dice=(1, 2)):
    r = np.zeros(32, np.int8)
    r[:24] = board
    r[24:26] = bar
    r[26:28] = off
    r[28] = player
    r[29:31] = dice
    return r


def board(**points):
    """board(p19=2, ...) by point number (1..24); + PLAYER1, - PLAYER2"""
    b = np.zeros(24, np.int8)
    for k, v in points.items():
        b[int(k[1:]) - 1] = v
    return b


def hand_picked():
    closed = board(p19=2, p20=2, p21=2, p22=2, p23=2, p24=2, p11=3, p1=-4, p2=-4, p3=-3, p4=-3)   # PLAYER2 on the bar shut out
    p2_home = board(p1=-2, p2=-2, p3=-2, p4=-2, p5=-2, p6=-2, p13=-3, p19=4, p20=4, p21=3, p22=3)
    bar_p2 = board(p19=3, p20=3, p21=3, p12=3, p6=3, p1=-5, p13=-5, p8=-3)
    return np.stack([
        rec_of(board(p24=1, p1=-5, p2=-5, p3=-5), off=(14, 0), player=0, dice=(3, 1)),            # PLAYER1 can win
        rec_of(board(p1=-1, p22=5, p23=5, p24=5), off=(0, 14), player=1, dice=(2, 2)),            # PLAYER2 can win
        rec_of(board(p24=2, p23=1, p1=-5, p2=-5, p3=-5), off=(12, 0), player=0, dice=(1, 1)),     # a double that bears off
        rec_of(closed, bar=(0, 1), player=0, dice=(2, 1)),                                       # opponent blocked after every move
        rec_of(closed, bar=(0, 1), player=0, dice=(4, 4)),
        rec_of(p2_home, bar=(1, 0), player=0, dice=(3, 5)),                                      # blocked non-double: no candidate
        rec_of(p2_home, bar=(1, 0), player=0, dice=(2, 2)),                                      # blocked double: one candidate
        rec_of(bar_p2, bar=(0, 2), player=1, dice=(6, 3)),                                       # mover on the bar
        rec_of(bar_p2, bar=(0, 2), player=1, dice=(1, 1)),
        rec_of(START, player=0, dice=(3, 3)),                                                    # big opening double
    ])


# ------------------------------------------------------------------ CPU: the restatement against the spec, restated in torch

def test_twoply_oracle_matches_a_torch_restatement(orc, golden):
    import torch
    from bgx.model import TDLGammonModel, encode_rows
    from bgx.synth import make_queries
    W1, b1, w2, b2 = w = golden_weights(golden("model.npz"), "trained")
    m = TDLGammonModel()
    m.load_state_dict({"fc1.weight": torch.from_numpy(W1), "fc1.bias": torch.from_numpy(b1),
                       "fc2.weight": torch.from_numpy(w2), "fc2.bias": torch.from_numpy(b2)})

    def V(states, turn):
        with torch.no_grad():
            return m(torch.from_numpy(encode_rows(np.asarray(states, np.int64), turn))).squeeze(1).numpy()

    q = np.concatenate([hand_picked(), make_queries(22, seed=99)[0]])
    ref = twoply_batch(orc, w, q)
    seen_win = seen_blocked_nd = seen_blocked_dbl = 0
    for rec, o in zip(q, ref):
        p = int(rec[28])
        mv, ln, st = orc.turn_sequences(rec[:28].astype(np.int32), p, int(rec[29]), int(rec[30]))
        cands, firsts = [], []
        for i in range(len(ln)):                                  # distinct afterstates, first appearance
            if not any(np.array_equal(st[i], c) for c in cands):
                cands.append(st[i])
                firsts.append(i)
        assert len(cands) == len(o["states"])
        for c, f, s, mvo, lno in zip(cands, firsts, o["states"], o["moves"], o["lens"]):
            assert np.array_equal(c, s) and np.array_equal(mv[f], mvo) and ln[f] == lno
        if not cands:
            assert o["pick"] == -1 and np.isnan(o["value"])
            continue
        if any(c[26 + p] == 15 for c in cands):
            seen_win += 1
            assert o["pick"] == [c[26 + p] == 15 for c in cands].index(True) and o["value"] == (0.0 if p else 1.0)
            continue
        v1 = V(np.stack(cands), p)
        assert np.allclose(v1, o["v1"], rtol=1e-5, atol=0)
        for j, A in enumerate(cands):
            acc = 0.0
            for (a, b), wt in zip(ROLLS, WEIGHTS):
                rmv, rln, rst = orc.turn_sequences(A, 1 - p, a, b)
                if len(rln) == 0 or rln.max() == 0:              # the opponent cannot move: the position stays
                    seen_blocked_nd += len(rln) == 0
                    seen_blocked_dbl += len(rln) > 0
                    R = V(A[None], 1 - p)[0]
                else:                                            # the opponent's greedy reply (model.py:205-213)
                    vals = V(rst, 1 - p)
                    R = vals[int(np.argmin(vals) if p == 0 else np.argmax(vals))]
                acc += wt * float(R)
            e2 = acc / 36.0
            assert abs(o["e2"][j] - e2) <= 1e-5 * abs(e2), (j, o["e2"][j], e2)
    assert seen_win >= 3 and seen_blocked_nd > 0 and seen_blocked_dbl > 0


# ------------------------------------------------------------------ GPU

@pytest.fixture(scope="module")
def eng():
    from bgx.engine import BatchEngine
    e = BatchEngine(0)
    yield e
    e.close()


def replay(orc, rec, moves, moves_len):
    s = rec[:28].astype(np.int32)
    for j in range(moves_len):
        o, d = (int(x) for x in moves[j])
        ok, _, s = orc.try_move(s, int(rec[28]), abs(o - d), o, d)
        assert ok
    return s


def check_against_oracle(orc, w, q, out, ref, K):
    """Every query: the engine's pick is the restatement's or a near-tie; values, counts and sequences as the spec says.
    Returns the number of near-ties."""
    soft = 0
    for i, (rec, o) in enumerate(zip(q, ref)):
        p = int(rec[28])
        U = len(o["lens"])
        assert out["n_candidates"][i] == U and out["n_expanded"][i] == o["n_expanded"], i
        ch = out["chosen"][i]
        assert np.array_equal(replay(orc, rec, out["moves"][i], out["moves_len"][i]), ch[:28].astype(np.int32)), i
        if U == 0:
            assert np.array_equal(ch[:28], rec[:28]) and ch[28] == p and ch[31] == 0 and np.isnan(out["value"][i])
            continue
        assert ch[28] == p and ch[31] == (out["moves_len"][i] > 0)
        j = [k for k in range(U) if np.array_equal(o["states"][k], ch[:28])]
        assert len(j) == 1, i
        j = j[0]
        if o["wins"].any():
            assert j == o["pick"] and out["value"][i] == (0.0 if p else 1.0), i
        else:
            e2 = o["e2"]
            if not o["expanded"][j]:                             # the engine expanded another top-K set: value it fully
                e2 = twoply_batch(orc, w, q[i:i + 1], 0)[0]["e2"]
                key = np.sort(-o["v1"] if p else o["v1"])[::-1]
                assert abs(key[K - 1] - key[K]) <= 1e-5 * abs(key[K - 1]), i
            assert abs(out["value"][i] - e2[j]) <= 1e-5 * abs(e2[j]), (i, out["value"][i], e2[j])
            if j != o["pick"]:
                soft += 1
                if o["expanded"][j]:
                    assert abs(e2[j] - e2[o["pick"]]) <= 1e-5 * abs(e2[o["pick"]]), i
        if j == o["pick"]:
            assert out["moves_len"][i] == o["lens"][j] and np.array_equal(out["moves"][i], o["moves"][j]), i
    return soft


@pytest.mark.gpu
@pytest.mark.parametrize("K", [0, 4])
@pytest.mark.parametrize("tag", ["rand", "trained"])
def test_twoply_vs_oracle(eng, orc, golden, tag, K):
    from bgx.synth import make_queries
    w = golden_weights(golden("model.npz"), tag)
    eng.set_weights(*w)
    q, _ = make_queries(2000, seed=4711)
    out = eng.select_moves_2ply_host(q, K)
    _, U, _ = eng.enumerate_summary_host(q)
    assert np.array_equal(out["n_candidates"], U)
    ref = twoply_batch(orc, w, q, K)
    soft = check_against_oracle(orc, w, q, out, ref, K)
    assert soft <= (0.10 if tag == "rand" else 0.01) * len(q), soft


@pytest.mark.gpu
def test_twoply_k1_is_select_moves(eng, golden):
    from bgx.synth import make_queries
    eng.set_weights(*golden_weights(golden("model.npz"), "trained"))
    q, _ = make_queries(30000, seed=1234)
    q = q[q[np.arange(len(q)), 26 + q[:, 28].astype(np.int64)] <= 10][:20000]   # at most 4 checkers borne off in a turn: no win
    assert len(q) == 20000
    one = eng.select_moves_host(q)
    two = eng.select_moves_2ply_host(q, 1)
    p = q[:, 28].astype(np.int64)
    assert (two["chosen"][np.arange(len(q)), 26 + p] != 15).all()
    for k in ("chosen", "moves", "moves_len"):
        assert np.array_equal(one[k], two[k]), k
    assert np.array_equal(two["n_expanded"], (two["n_candidates"] > 0).astype(np.int32))
    assert np.array_equal(two["value"] != two["value"], one["value"] != one["value"])      # NaN exactly without a sequence


@pytest.mark.gpu
def test_twoply_edge_cases(eng, orc, golden):
    from bgx import lib as L
    from bgx.engine import BatchEngine
    w = golden_weights(golden("model.npz"), "trained")
    eng.set_weights(*w)
    hp = hand_picked()
    out = eng.select_moves_2ply_host(hp, 0)
    # winning candidates: taken, exactly 1 / 0, nothing expanded
    for i in (0, 1, 2):
        p = int(hp[i, 28])
        assert out["chosen"][i, 26 + p] == 15 and out["value"][i] == (0.0 if p else 1.0) and out["n_expanded"][i] == 0
        assert np.array_equal(replay(orc, hp[i], out["moves"][i], out["moves_len"][i]), out["chosen"][i, :28].astype(np.int32))
    # blocked non-double: the position back, nothing played, NaN
    assert np.array_equal(out["chosen"][5, :28], hp[5, :28]) and out["chosen"][5, 28] == 0 and out["chosen"][5, 31] == 0
    assert np.isnan(out["value"][5]) and out["n_candidates"][5] == 0 and out["moves_len"][5] == 0
    # blocked double: one candidate, the empty sequence, its E2
    assert out["n_candidates"][6] == 1 and out["n_expanded"][6] == 1 and out["moves_len"][6] == 0 and out["chosen"][6, 31] == 0
    assert np.array_equal(out["chosen"][6, :28], hp[6, :28]) and np.isfinite(out["value"][6])
    ref = twoply_batch(orc, w, hp, 0)
    assert abs(out["value"][6] - ref[6]["value"]) <= 1e-5 * abs(ref[6]["value"])
    # arguments
    lib = eng._lib
    with pytest.raises(L.BgxError):
        L.check(lib.bgx_select_moves_2ply_host(eng._h, hp.ctypes.data, -1, 0, None, None, None, None, None, None))
    with pytest.raises(L.BgxError):
        L.check(lib.bgx_select_moves_2ply_host(eng._h, hp.ctypes.data, len(hp), -1, None, None, None, None, None, None))
    with pytest.raises(L.BgxError):
        eng.set_option("twoply_chunk", -5)
    L.check(lib.bgx_select_moves_2ply_host(eng._h, hp.ctypes.data, 0, 0, None, None, None, None, None, None))
    fresh = BatchEngine(0)
    try:
        with pytest.raises(L.BgxError) as e:
            fresh.select_moves_2ply_host(hp)
        assert e.value.code == L.E_STATE
    finally:
        fresh.close()


@pytest.mark.gpu
@pytest.mark.parametrize("K", [0, 3])
def test_twoply_is_a_pure_function_of_the_query(eng, golden, K):
    from bgx.synth import make_queries
    eng.set_weights(*golden_weights(golden("model.npz"), "trained"))
    q, _ = make_queries(3000, seed=8080)
    keys = ("chosen", "moves", "moves_len", "value", "n_candidates", "n_expanded")

    def same(a, b, idx=None):
        for k in keys:
            x = a[k] if idx is None else a[k][idx]
            if k == "value":
                assert np.array_equal(b[k].view(np.uint32), x.view(np.uint32)), k
            else:
                assert np.array_equal(b[k], x), k

    whole = eng.select_moves_2ply_host(q, K)
    few = np.flatnonzero(whole["n_candidates"] > 20)[:48]
    same(whole, eng.select_moves_2ply_host(q[few], K), few)                   # alone
    big = np.concatenate([make_queries(20000, seed=5)[0], q])
    same(whole, {k: v[20000:] for k, v in eng.select_moves_2ply_host(big, K).items()})
    perm = np.random.default_rng(3).permutation(len(q))
    same(whole, eng.select_moves_2ply_host(q[perm], K), perm)
    n_replies = int(whole["n_expanded"].sum()) * 21
    eng.set_option("twoply_chunk", 21 * 97)
    try:
        assert n_replies > 3 * 21 * 97
        same(whole, eng.select_moves_2ply_host(q, K))
    finally:
        eng.set_option("twoply_chunk", 0)


@pytest.mark.gpu
def test_twoply_surfaces_agree(eng, golden):
    import torch
    import backgammon_env as bg
    from bgx.model import TDLGammonModel
    from bgx.synth import make_queries
    W1, b1, w2, b2 = w = golden_weights(golden("model.npz"), "trained")
    eng.set_weights(*w)
    q, _ = make_queries(2000, seed=77)
    host = eng.select_moves_2ply_host(q, 2)
    dev = {k: torch.zeros(v.shape, dtype=getattr(torch, str(v.dtype)), device="cuda") for k, v in host.items()}
    qd = torch.from_numpy(q).cuda()
    torch.cuda.synchronize()
    eng.select_moves_2ply(qd, 2, **dev)
    eng.synchronize()
    for k in host:
        assert np.array_equal(dev[k].cpu().numpy().view(np.uint8), host[k].view(np.uint8)), k
    be = bg.BatchEngine(0)
    be.set_weights(*w)
    mm = be.make_moves_2ply(q, 2)
    for k in host:
        assert np.array_equal(np.asarray(mm[k]).view(np.uint8), host[k].view(np.uint8)), k
    # make_moves_batch(plies=2) plays the engine's sequences on compat Games
    m = TDLGammonModel()
    m.load_state_dict({"fc1.weight": torch.from_numpy(W1), "fc1.bias": torch.from_numpy(b1),
                       "fc2.weight": torch.from_numpy(w2), "fc2.bias": torch.from_numpy(b2)})
    with pytest.raises(ValueError):
        m.make_moves_batch([bg.Game(0)], epsilon=0.1, plies=2)
    rng = np.random.default_rng(5)
    games = [bg.Game(i % 2) for i in range(48)]
    for _ in range(8):
        q = np.zeros((len(games), 32), np.int8)
        for i, g in enumerate(games):
            d = rng.integers(1, 7, 2)
            g.setDice(int(d[0]), int(d[1]))
            q[i, :24] = g.getGameBoard()
            q[i, 24], q[i, 25] = g.getJailedCount(0), g.getJailedCount(1)
            q[i, 26], q[i, 27] = g.getBornOffCount(0), g.getBornOffCount(1)
            q[i, 28] = g.getTurn()
            q[i, 29:31] = g.get_last_dice()
        want = eng.select_moves_2ply_host(q, 3)
        seqs = m.make_moves_batch(games, plies=2, candidates=3)
        for i, g in enumerate(games):
            assert len(seqs[i]) == want["moves_len"][i]
            got = list(g.getGameBoard()) + [g.getJailedCount(0), g.getJailedCount(1), g.getBornOffCount(0), g.getBornOffCount(1)]
            assert np.array_equal(np.array(got), want["chosen"][i, :28].astype(np.int64)), i
            g.setTurn(1 - int(g.getTurn()))


@pytest.mark.gpu
def test_twoply_arena_games_replay_through_the_oracle(orc, golden):
    from bgx.evaluate import Arena, TwoPly
    gm = golden("model.npz")
    wt, wr = golden_weights(gm, "trained"), golden_weights(gm, "rand")
    n, K = 8, 4
    side = (np.arange(n) % 2).astype(np.int8)
    first = ((np.arange(n) // 2) % 2).astype(np.int8)
    arena = Arena(0)
    try:
        res = arena.play(TwoPly(wt, K), wr, side, first, seed=SEED, record=True)
    finally:
        arena.close()
    assert (res["winner"] >= 0).all()
    state = {i: None for i in range(n)}
    count = np.zeros(n, np.int64)
    two_q, two_ch, soft = [], [], 0
    for ply, idx, q, ch in res["log"]:
        for j, g in enumerate(idx):
            r = q[j]
            x = orc.philox(SEED, ply, int(g))
            assert (int(r[29]), int(r[30])) == (orc.die(x[0]), orc.die(x[1]))
            assert int(r[28]) == (int(first[g]) ^ (ply & 1))
            if state[g] is None:
                assert np.array_equal(r[:24], START) and not r[24:28].any()
            else:
                assert np.array_equal(r[:28], state[g])
            if int(r[28]) == int(side[g]):
                two_q.append(r)
                two_ch.append(ch[j])
            else:                                                    # the one-ply side: the oracle's greedy pick
                i0, after, v, _ = orc.greedy_ply(wr, r[:28].astype(np.int32), int(r[28]), r[29], r[30])
                if i0 >= 0 and not np.array_equal(ch[j, :28].astype(np.int32), after):
                    vg = orc.forward(wr, orc.encode(ch[j, :28].astype(np.int32)[None], int(r[28])))[0]
                    assert abs(vg - v) <= 1e-5 * abs(v)
                    soft += 1
            state[g] = ch[j, :28].copy()
            count[g] += 1
    two_q, two_ch = np.array(two_q), np.array(two_ch)
    ref = twoply_batch(orc, wt, two_q, K)
    for i, (r, o) in enumerate(zip(two_q, ref)):
        if o["pick"] < 0:
            assert np.array_equal(two_ch[i, :28], r[:28])
            continue
        j = [k for k in range(len(o["lens"])) if np.array_equal(o["states"][k], two_ch[i, :28])]
        assert len(j) == 1
        j = j[0]
        if j != o["pick"]:
            soft += 1
            e2 = twoply_batch(orc, wt, two_q[i:i + 1], 0)[0]["e2"]
            key = np.sort(-o["v1"] if r[28] else o["v1"])[::-1]
            assert (abs(e2[j] - e2[o["pick"]]) <= 1e-5 * abs(e2[o["pick"]]) or
                    (len(key) > K and abs(key[K - 1] - key[K]) <= 1e-5 * abs(key[K - 1]))), i
    assert soft <= 0.1 * count.sum()
    for g in range(n):
        assert orc.game_over(state[g].astype(np.int32)) == int(res["winner"][g])
        assert count[g] == res["plies"][g]


@pytest.mark.gpu
def test_twoply_plays_better_than_one_ply(golden):
    """4,096 games of the trained net looking one roll ahead against itself at one ply, sides and first mover alternated:
    the two-ply side wins more than half the games by three standard deviations."""
    from bgx.evaluate import Arena, TwoPly
    wt = golden_weights(golden("model.npz"), "trained")
    n = 4096
    i = np.arange(n)
    side = (i % 2).astype(np.int8)
    first = ((i // 2) % 2).astype(np.int8)
    arena = Arena(0)
    try:
        res = arena.play(TwoPly(wt), wt, side, first, seed=SEED)
    finally:
        arena.close()
    assert (res["winner"] >= 0).all()
    rate = float(np.mean(res["winner"] == side))
    print(f"two-ply vs one-ply win rate over {n} games: {rate:.4f}")
    assert rate >= 0.5 + 3 * 0.5 / np.sqrt(n), rate
