"""The fused ply kernels (k_select, k_selfplay) where a comparison with the oracle has no slack and the suite's other inputs
do not reach:
  A. tie nets - weights under which many distinct afterstates have bit-equal values, so the strict first-index arg-best, the
     sharing merge's "lower root origin" rule and the two-pass bookkeeping of a non-double decide the pick; the right answer is
     an integer fact about the enumeration, not a value within 1e-5;
  B. every launch configuration the kernels ship with (warps per CTA, unsorted queue, sharing policy, asynchronous lanes);
  C. partial exploration (0 < epsilon < 1), checked per decision, and self-play games that mix explored and greedy plies;
  D. launches long enough that the per-warp cache generation wraps (PlyCache::next_ply)."""
import numpy as np
import pytest

from conftest import golden_weights

SEED = 0x5EED2026
EPS = 0.3
EXPLORE_SEED = 20261020
INV_2_32 = np.float32(2.3283064365386963e-10)        # the kernels' 2^-32 (k_select, k_selfplay)
KEYS = ("chosen", "moves", "moves_len", "value", "n_seq")
TIE_NETS = ("flat", "off", "bar")
# columns (plus, minus) of the record whose difference the value of a tie net rises with, for PLAYER1
TIE_COLUMNS = {"flat": None, "off": (26, 27), "bar": (25, 24)}


# ------------------------------------------------------------------ tie nets and their integer rule

def tie_net(kind, seed=11):
    """Weights under which the value of an afterstate is a strictly monotone function of one integer, exactly.
      flat: W1 = 0, so V is one constant and every pick is sequence 0.
      off:  only the borne-off columns 196 / 197 (+ for PLAYER1, - for PLAYER2) and w2 > 0: V rises with PLAYER1's borne-off count
            and falls with PLAYER2's.
      bar:  only the bar columns 194 / 195, equal magnitude and opposite sign: V is a function of bar(PLAYER2) - bar(PLAYER1).
    Every weight is a dyadic number with few bits, so the oracle's fp32 sum over the 198 features and the kernels' fixed-point sum
    are exact: equal features give bit-equal values, and one checker more changes V by ~1e-2."""
    rng = np.random.default_rng(seed)
    W1 = np.zeros((128, 198), np.float32)
    b1 = (rng.integers(-64, 65, 128) / 64).astype(np.float32)
    if kind == "flat":
        w2 = (rng.integers(-32, 33, (1, 128)) / 256).astype(np.float32)
        b2 = np.array([0.25], np.float32)
        return W1, b1, w2, b2
    w2 = (rng.integers(1, 33, (1, 128)) / 512).astype(np.float32)
    if kind == "off":
        W1[:, 196] = rng.integers(32, 97, 128) / 64
        W1[:, 197] = -rng.integers(32, 97, 128) / 64
    else:
        c = rng.integers(16, 49, 128) / 64
        W1[:, 194] = -c
        W1[:, 195] = c
    b2 = np.array([-np.round(0.5 * w2.sum() * 64) / 64], np.float32)      # V near 1/2: far from saturation
    return W1, b1, w2, b2


def signed_feature(kind, states, player):
    """The integer a tie net's value rises with, from the mover's side (the mover maximises it)."""
    st = np.asarray(states, np.int64)
    if TIE_COLUMNS[kind] is None:
        return np.zeros(len(st), np.int64)
    a, b = TIE_COLUMNS[kind]
    return (1 - 2 * int(player)) * (st[:, a] - st[:, b])


def integer_rule(orc, queries, kinds=TIE_NETS, count_ties=False):
    """The pick of the greedy ply under each tie net, from the oracle's ordered sequence list: the first sequence whose afterstate
    maximises the mover's signed feature.  -> {"n_seq": int64[n], kind: {"pick", "after", "moves", "moves_len"[, "n_best"]}};
    pick -1 and the position itself where there is no sequence; n_best: how many distinct afterstates share the best feature."""
    n = len(queries)
    out = {"n_seq": np.zeros(n, np.int64)}
    for k in kinds:
        out[k] = {"pick": np.full(n, -1, np.int64), "after": queries[:, :28].astype(np.int8).copy(),
                  "moves": np.zeros((n, 4, 2), np.int8), "moves_len": np.zeros(n, np.int8)}
        if count_ties:
            out[k]["n_best"] = np.zeros(n, np.int64)        # distinct afterstates of the best key
    for i, r in enumerate(queries):
        p = int(r[28])
        mv, ln, st = orc.turn_sequences(r[:28].astype(np.int32), p, int(r[29]), int(r[30]))
        out["n_seq"][i] = len(ln)
        if len(ln) == 0:
            continue
        rows = np.ascontiguousarray(st).view(np.dtype((np.void, 28 * 4))).ravel() if count_ties else None
        for k in kinds:
            key = signed_feature(k, st, p)
            j = int(np.argmax(key))                          # the first index of the maximum
            o = out[k]
            o["pick"][i] = j
            o["after"][i] = st[j]
            o["moves"][i] = mv[j]
            o["moves_len"][i] = ln[j]
            if count_ties:
                o["n_best"][i] = len(set(rows[key == key[j]].tolist()))
    return out


def forward64(w, orc, states, players):
    """V of afterstates in float64 (model.py:63-67) on the oracle's encoding."""
    W1, b1, w2, b2 = (np.asarray(a, np.float64) for a in w)
    v = np.zeros(len(states))
    for t in (0, 1):
        m = players == t
        if m.any():
            X = orc.encode(np.asarray(states, np.int32)[m], t).astype(np.float64)
            h = 1.0 / (1.0 + np.exp(-(X @ W1.reshape(128, 198).T + b1)))
            v[m] = 1.0 / (1.0 + np.exp(-(h @ w2.reshape(-1) + b2[0])))
    return v


def explore_draws(orc, seed, c0, c1, eps):
    """k_select / k_selfplay's exploration draw Philox(seed; c0, c1, 0, 2): (explore?, x1) per counter pair."""
    ex = np.zeros(len(c1), bool)
    x1 = np.zeros(len(c1), np.uint64)
    for i, (a, b) in enumerate(zip(c0, c1)):
        x = orc.philox(seed, int(a), int(b) & 0xFFFFFFFF, int(b) >> 32, 2)
        ex[i] = np.float32(x[0]) * INV_2_32 < np.float32(eps)
        x1[i] = x[1]
    return ex, x1


# ------------------------------------------------------------------ CPU: the integer rule is the oracle's greedy ply

@pytest.mark.parametrize("kind", TIE_NETS)
def test_tie_net_integer_rule_is_the_oracle(orc, kind):
    """On 20,000 seeded queries the oracle's greedy ply (first-index arg-best over V, model.py:205-213) under a tie net is the
    integer rule, sequence for sequence; the nets are exact (equal features: bit-equal V; unequal: far apart); and the inputs
    really tie: many queries have several distinct best afterstates, the first of them not sequence 0, big doubles included."""
    from bgx.synth import make_queries
    w = tie_net(kind)
    q, _ = make_queries(20000, seed=606)
    ref = integer_rule(orc, q, (kind,), count_ties=True)
    g = orc.greedy_batch(w, q)
    o = ref[kind]
    has = ref["n_seq"] > 0
    assert np.array_equal(g["n_seq"], ref["n_seq"])
    assert np.array_equal(g["after"][has], o["after"][has])
    assert np.array_equal(g["moves"][has], o["moves"][has]) and np.array_equal(g["moves_len"][has], o["moves_len"][has])
    # the premise: within a turn V is a strictly monotone function of the signed feature, exactly
    for i in range(0, len(q), 10):
        r = q[i]
        p = int(r[28])
        _, _, st = orc.turn_sequences(r[:28].astype(np.int32), p, int(r[29]), int(r[30]))
        if len(st) < 2:
            continue
        v = orc.forward(w, orc.encode(st, p)).astype(np.float64) * (1 - 2 * p)
        key = signed_feature(kind, st, p)
        for a in np.unique(key):
            assert len(np.unique(v[key == a])) == 1, (i, a)                       # equal features: bit-equal V
        s = np.unique(key)
        if len(s) > 1:
            vs = np.array([v[key == a][0] for a in s])
            assert (np.diff(vs) > 1e-4).all(), (i, vs)                             # unequal: ordered, far beyond 1e-5
    # measured on these queries: 67 / 53 / 62 % tied, 0 / 7.4 / 6.4 % tied with a later first best; of the 388 big doubles 388 /
    # 383 / 378 tied, 0 / 3 / 93 with a later first best (flat / off / bar)
    big = (q[:, 29] == q[:, 30]) & (ref["n_seq"] > 500)
    tied = o["n_best"] >= 2
    assert tied.mean() > 0.45, tied.mean()
    assert big.sum() > 300 and (tied & big).sum() > 0.95 * big.sum()
    hard = tied & (o["pick"] > 0)
    if kind == "flat":
        assert (o["pick"][has] == 0).all()
    else:
        assert hard.mean() > 0.05, hard.mean()
    if kind == "bar":
        assert (hard & big).sum() >= 50, (hard & big).sum()


# ------------------------------------------------------------------ GPU fixtures

@pytest.fixture(scope="module")
def eng():
    from bgx.engine import BatchEngine
    e = BatchEngine(0)
    yield e
    e.close()


@pytest.fixture
def fresh():
    """An engine of the test's own, so that options set on it never leak into other tests."""
    from bgx.engine import BatchEngine
    e = BatchEngine(0)
    yield e
    e.close()


@pytest.fixture(scope="module")
def large():
    """The 60,000 queries of test_select_moves_large_sample_vs_oracle."""
    from bgx.synth import make_queries
    return make_queries(60000, seed=777)[0]


@pytest.fixture(scope="module")
def rules(orc, large):
    return integer_rule(orc, large)


def weights_of(golden, net):
    return golden_weights(golden("model.npz"), net) if net in ("trained", "rand") else tie_net(net)


def assert_same(got, want, keys=KEYS, idx=None, what=""):
    for k in keys:
        w = want[k] if idx is None else want[k][idx]
        if k == "value":
            assert np.array_equal(got[k].view(np.uint32), w.view(np.uint32)), (what, k)
        else:
            assert np.array_equal(got[k], w), (what, k, int(np.sum(np.any((got[k] != w).reshape(len(w), -1), 1))))


def check_integer_rule(orc, w, q, out, ref, kind):
    """No near-tie allowance: afterstate, reported sequence and N are the integer rule's; V is the float64 forward's within 1e-5."""
    o = ref[kind]
    n = ref["n_seq"]
    has = n > 0
    assert np.array_equal(out["n_seq"].astype(np.int64), n)
    bad = np.flatnonzero(~(out["chosen"][:, :28] == o["after"]).all(1))
    assert bad.size == 0, (kind, "afterstate", bad.size, bad[:8])
    assert (out["chosen"][:, 28] == q[:, 28]).all()
    assert np.array_equal(out["moves_len"], o["moves_len"])
    bad = np.flatnonzero(has & ~(out["moves"] == o["moves"]).reshape(len(q), -1).all(1))
    assert bad.size == 0, (kind, "sequence", bad.size, bad[:8])
    assert np.isnan(out["value"][~has]).all()
    v64 = forward64(w, orc, out["chosen"][has, :28], q[has, 28])
    assert (np.abs(out["value"][has] - v64) <= 1e-5 * np.abs(v64)).all(), kind


# ------------------------------------------------------------------ A. tie nets on the GPU

@pytest.mark.gpu
@pytest.mark.parametrize("kind", TIE_NETS)
def test_select_moves_tie_nets_are_the_integer_rule(eng, orc, large, rules, kind):
    w = tie_net(kind)
    eng.set_weights(*w)
    out = eng.select_moves_host(large)
    check_integer_rule(orc, w, large, out, rules, kind)
    if kind == "flat":
        v = out["value"][rules["n_seq"] > 0]
        assert (v.view(np.uint32) == v[0].view(np.uint32)).all()                 # one constant


@pytest.mark.gpu
@pytest.mark.parametrize("kind", TIE_NETS)
def test_tie_nets_on_big_doubles_under_sharing(eng, fresh, orc, large, rules, kind):
    """Big doubles are walked by several warps of a CTA and merged by "better value, then lower root origin": alone (64 queries
    on the whole GPU: every sub-tree that can be taken is taken) and, on a fresh engine, every double of the sample with the
    giant threshold at the publishing threshold (every published double is helped at once)."""
    w = tie_net(kind)
    dbl = large[:, 29] == large[:, 30]
    big = np.flatnonzero(dbl & (rules["n_seq"] > 500))[:64]
    assert big.size == 64
    sub = {"n_seq": rules["n_seq"][big], kind: {k: v[big] for k, v in rules[kind].items()}}
    eng.set_weights(*w)
    check_integer_rule(orc, w, large[big], eng.select_moves_host(large[big]), sub, kind)
    fresh.set_weights(*w)
    fresh.set_option("select_giant_min", 4)                    # kStealMinChildren
    alld = np.flatnonzero(dbl)
    sub = {"n_seq": rules["n_seq"][alld], kind: {k: v[alld] for k, v in rules[kind].items()}}
    check_integer_rule(orc, w, large[alld], fresh.select_moves_host(large[alld]), sub, kind)


def restart_loop_matches_population(eng, n, plies):
    """bgx_selfplay_step(plies) on n slots = `plies` host-driven bgx_play_ply_restart_host_async steps (one k_select per ply),
    bit for bit: records, ply numbers, game ids, games finished and PLAYER1 wins."""
    from bgx import host as H
    from bgx.lib import FIRST_PARITY
    from bgx.synth import START_BOARD
    eng.selfplay_init(n, first_id=0, id_stride=n, seed=SEED, first_mover=FIRST_PARITY, traj_cap=0)
    st = eng.selfplay_step(plies)
    want_rec, want_ply, want_gid = eng.selfplay_read()
    gid = np.arange(n, dtype=np.int64)
    ply = np.zeros(n, np.int32)
    fresh = np.zeros((n, 32), np.int8)
    fresh[:, :24] = START_BOARD
    fresh[:, 28] = (gid & 1) ^ 1                           # bgx_advance_host flips the mover and rolls ply 0
    bufs = [H.advance(fresh, fresh.copy(), SEED, ply, gid), np.zeros((n, 32), np.int8)]
    win = np.zeros(n, np.int8)
    finished = p1 = 0
    cuts = [0, n // 3, n // 3 + 1, n]
    for step in range(plies):
        a, b = bufs[step & 1], bufs[1 - (step & 1)]
        for lane, (lo, hi) in enumerate(zip(cuts[:-1], cuts[1:])):
            eng.play_ply_restart_host_async(lane, a[lo:hi], ply[lo:hi], gid[lo:hi], n, b[lo:hi], win[lo:hi],
                                            first_mover=FIRST_PARITY, dice_seed=SEED)
        for lane in range(3):
            eng.wait(lane)
        finished += int((win >= 0).sum())
        p1 += int((win == 0).sum())
    got = bufs[plies & 1]
    assert np.array_equal(ply, want_ply) and np.array_equal(gid, want_gid)
    assert np.array_equal(got[:, :29], want_rec[:, :29])
    assert finished == st["games_finished"] and p1 == st["p1_wins"]
    return st


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["off", "bar"])
def test_selfplay_tie_nets_are_the_host_driven_loop(eng, kind):
    """k_selfplay under a tie net (its picks carried from ply to ply, its root pre-activation carried too) = the host-driven
    loop of k_select launches, which test_select_moves_tie_nets_are_the_integer_rule pins to the integer rule."""
    eng.set_weights(*tie_net(kind))
    restart_loop_matches_population(eng, 2000, 150)


@pytest.mark.gpu
@pytest.mark.parametrize("K", [0, 4])
def test_twoply_flat_net(eng, orc, K):
    """Two-ply under the flat net: every expanded candidate is worth exactly the constant V (every reply, blocked or not, is V),
    so the pick is candidate 0 - or the first winning candidate, worth exactly 1 / 0 - and the counts are the spec's."""
    from bgx.synth import make_queries
    from twoply_ref import candidates, twoply_batch
    w = tie_net("flat")
    eng.set_weights(*w)
    q, _ = make_queries(3000, seed=4712)
    out = eng.select_moves_2ply_host(q, K)
    one = eng.select_moves_host(q)
    V = one["value"][one["n_seq"] > 0][0]
    v64 = forward64(w, orc, q[:1, :28], q[:1, 28])[0]
    assert abs(V - v64) <= 1e-5 * v64
    wins_seen = 0
    for i, r in enumerate(q):
        p = int(r[28])
        st, mv, ln = candidates(orc, r)
        U = len(ln)
        assert out["n_candidates"][i] == U, i
        if U == 0:
            assert np.isnan(out["value"][i]) and out["n_expanded"][i] == 0 and np.array_equal(out["chosen"][i, :28], r[:28])
            continue
        wins = st[:, 26 + p] == 15
        j = int(np.argmax(wins)) if wins.any() else 0
        wins_seen += bool(wins.any())
        assert np.array_equal(out["chosen"][i, :28], st[j].astype(np.int8)), i
        assert out["moves_len"][i] == ln[j] and np.array_equal(out["moves"][i], mv[j]), i
        if wins.any():
            assert out["value"][i] == (0.0 if p else 1.0) and out["n_expanded"][i] == 0, i
        else:
            assert out["value"][i].view(np.uint32) == V.view(np.uint32), i
            assert out["n_expanded"][i] == (U if K == 0 else min(K, U)), i
    assert wins_seen > 100
    for i, o in enumerate(twoply_batch(orc, w, q[:120], K)):                   # the CPU restatement: ~2,000 replies per query
        assert out["n_expanded"][i] == o["n_expanded"]
        if o["pick"] < 0:
            continue
        assert np.array_equal(out["chosen"][i, :28], o["states"][o["pick"]].astype(np.int8)), i
        assert abs(out["value"][i] - o["value"]) <= 1e-5 * abs(o["value"]), i


# ------------------------------------------------------------------ B. launch-configuration invariance

SELECT_CONFIGS = {
    "warps16": {"select_warps": 16},
    "warps24": {"select_warps": 24},
    "warps32": {"select_warps": 32},
    "unsorted_queue": {"select_order_max": 0},
    "all_urgent": {"select_giant_min": 4},
    "end_of_queue_help": {"select_giant_min": 99, "select_urgent_min": 99},
    "urgent_from_start": {"select_urgent_min": 4, "select_urgent_from_pct": 0},
}


@pytest.fixture(scope="module")
def defaults(eng, orc, golden, large):
    """Default-configuration k_select results on the 60,000 queries per (net, epsilon), and which queries explored.  At epsilon 0
    they are pinned by test_select_moves_large_sample_vs_oracle (trained net, same queries) and by
    test_select_moves_tie_nets_are_the_integer_rule (off net); at 0.3 by test_select_moves_partial_exploration_per_query."""
    res = {}
    for net in ("trained", "off"):
        eng.set_weights(*weights_of(golden, net))
        for eps in (0.0, EPS):
            res[net, eps] = eng.select_moves_host(large, epsilon=eps, seed=EXPLORE_SEED)
    res["explore"], res["x1"] = explore_draws(orc, EXPLORE_SEED, np.zeros(len(large)), np.arange(len(large)), EPS)
    res["U"] = eng.enumerate_summary_host(large)[1]
    return res


def check_n_scored(out, defaults, explored):
    """Every distinct afterstate of a greedy query is scored at least once, and nothing is scored that is not a sequence's end;
    an explored query scores nothing."""
    s, n, U = out["n_scored"], out["n_seq"], defaults["U"]
    g = ~explored
    assert (s[g] >= U[g]).all() and (s[g] <= n[g]).all()
    assert (s[explored] == 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("config,eps", [(c, 0.0) for c in SELECT_CONFIGS] + [(c, EPS) for c in SELECT_CONFIGS if c.startswith("warps")])
@pytest.mark.parametrize("net", ["trained", "off"])
def test_select_moves_do_not_depend_on_the_launch_configuration(fresh, golden, large, defaults, net, config, eps):
    fresh.set_weights(*weights_of(golden, net))
    for k, v in SELECT_CONFIGS[config].items():
        fresh.set_option(k, v)
    out = fresh.select_moves_host(large, epsilon=eps, seed=EXPLORE_SEED)
    assert_same(out, defaults[net, eps], what=(net, config, eps))
    check_n_scored(out, defaults, defaults["explore"] if eps > 0 else np.zeros(len(large), bool))


@pytest.mark.gpu
@pytest.mark.parametrize("grid", [1, 0])
@pytest.mark.parametrize("net", ["trained", "off"])
def test_select_moves_on_a_lane_do_not_depend_on_its_grid(fresh, golden, large, defaults, net, grid):
    import torch
    fresh.set_weights(*weights_of(golden, net))
    fresh.set_option("select_lane_grid", grid)
    want = defaults[net, 0.0]
    pin = {k: torch.from_numpy(np.zeros_like(want[k])).pin_memory().numpy() for k in KEYS + ("n_scored",)}
    qp = torch.from_numpy(large.copy()).pin_memory().numpy()
    fresh.select_moves_host_async(1, qp, pin)
    fresh.wait(1)
    assert_same(pin, want, what=(net, grid))
    check_n_scored(pin, defaults, np.zeros(len(large), bool))


@pytest.mark.gpu
@pytest.mark.parametrize("warps", [16, 32])
@pytest.mark.parametrize("net", ["trained", "off"])
def test_twoply_does_not_depend_on_the_select_warps(eng, fresh, golden, large, net, warps):
    w = weights_of(golden, net)
    q = large[:10000]
    eng.set_weights(*w)
    want = eng.select_moves_2ply_host(q, 0)
    fresh.set_weights(*w)
    fresh.set_option("select_warps", warps)
    got = fresh.select_moves_2ply_host(q, 0)
    assert_same(got, want, ("chosen", "moves", "moves_len", "value", "n_candidates", "n_expanded"), what=(net, warps))


SELFPLAY_SLOTS = 1024


def selfplay_run(e, eps):
    """A step of 60 plies (restarts in place), then a round to the end of every game, with trajectories."""
    e.selfplay_init(SELFPLAY_SLOTS, first_id=0, id_stride=SELFPLAY_SLOTS, seed=SEED, traj_cap=1024, record_chosen=True)
    s1 = e.selfplay_step(60, epsilon=eps)
    s2 = e.selfplay_round(epsilon=eps)
    rec, ply, gid = e.selfplay_read()
    trajs = [e.export_trajectory(s) for s in range(0, SELFPLAY_SLOTS, 41)]
    return s1, s2, (rec, ply, gid), trajs


@pytest.fixture(scope="module")
def selfplay_defaults(eng, golden):
    eng.set_weights(*golden_weights(golden("model.npz"), "trained"))
    return {eps: selfplay_run(eng, eps) for eps in (0.0, EPS)}


@pytest.mark.gpu
@pytest.mark.parametrize("eps", [0.0, EPS])
@pytest.mark.parametrize("warps", [16, 24, 32])
def test_selfplay_does_not_depend_on_the_warps_per_cta(fresh, golden, selfplay_defaults, warps, eps):
    fresh.set_weights(*golden_weights(golden("model.npz"), "trained"))
    fresh.set_option("selfplay_warps", warps)
    s1, s2, read, trajs = selfplay_run(fresh, eps)
    w1, w2, wread, wtrajs = selfplay_defaults[eps]
    for a, b in ((s1, w1), (s2, w2)):
        for k in ("plies", "sequences", "games_finished", "p1_wins", "truncated"):
            assert a[k] == b[k], (k, a[k], b[k])
    assert w2["truncated"] == 0 and w2["games_finished"] == SELFPLAY_SLOTS
    for a, b in zip(read, wread):
        assert np.array_equal(a, b)
    for (p, c), (wp, wc) in zip(trajs, wtrajs):
        assert np.array_equal(p, wp) and np.array_equal(c, wc)


# ------------------------------------------------------------------ C. partial exploration, per decision

@pytest.mark.gpu
def test_select_moves_partial_exploration_per_query(eng, orc, golden, large, defaults):
    """epsilon = 0.3: a query explores iff x0 * 2^-32 < epsilon (fp32) for Philox(seed; 0, q, 0, 2), and then takes sequence
    (x1 * N) >> 32 in reference order; every other query is the greedy ply, bit for bit."""
    out, greedy = defaults["trained", EPS], defaults["trained", 0.0]
    ex = defaults["explore"]
    assert 0.25 < ex.mean() < 0.35
    assert_same({k: v[~ex] for k, v in out.items()}, greedy, idx=~ex, what="greedy queries")
    for i in np.flatnonzero(ex):
        r = large[i]
        mv, ln, st = orc.turn_sequences(r[:28].astype(np.int32), int(r[28]), int(r[29]), int(r[30]))
        assert out["n_seq"][i] == len(ln) and np.isnan(out["value"][i]) and out["n_scored"][i] == 0, i
        if len(ln) == 0:
            assert np.array_equal(out["chosen"][i, :28], r[:28]) and out["moves_len"][i] == 0, i
            continue
        k = (int(defaults["x1"][i]) * len(ln)) >> 32
        assert np.array_equal(out["chosen"][i, :28], st[k].astype(np.int8)), i
        assert out["moves_len"][i] == ln[k] and np.array_equal(out["moves"][i], mv[k]), i


@pytest.mark.gpu
def test_selfplay_partial_exploration_per_ply(eng, orc, golden):
    """A self-play round at epsilon = 0.3, every ply of 256 games: an explored ply (draw of (ply, game id, stream 2)) takes the
    drawn sequence; a greedy ply is select_moves on its pre-move record, bit for bit - including the greedy plies right after
    explored ones, where the root pre-activation carried from the previous ply must not be used."""
    w = golden_weights(golden("model.npz"), "trained")
    eng.set_weights(*w)
    n = 256
    eng.selfplay_init(n, first_id=3000, id_stride=n, seed=SEED, traj_cap=2048, record_chosen=True)
    st = eng.selfplay_round(epsilon=EPS)
    assert st["games_finished"] == n and st["truncated"] == 0
    _, _, gid = eng.selfplay_read()
    pre_all, cho_all, ex_all, x1_all, after_ex = [], [], [], [], []
    for slot in range(n):
        pre, cho = eng.export_trajectory(slot)
        T = len(pre)
        assert T > 0
        assert np.array_equal(pre[1:, :28], cho[:-1, :28])
        ex, x1 = explore_draws(orc, SEED, np.arange(T), np.full(T, gid[slot]), EPS)
        pre_all.append(pre); cho_all.append(cho); ex_all.append(ex); x1_all.append(x1)
        after_ex.append(np.concatenate([[False], ex[:-1]]) & ~ex)
    pre, cho, ex, x1, after_ex = (np.concatenate(a) for a in (pre_all, cho_all, ex_all, x1_all, after_ex))
    assert 0.25 < ex.mean() < 0.35 and after_ex.sum() > 2000
    g = eng.select_moves_host(pre[~ex])
    assert np.array_equal(cho[~ex, :28], g["chosen"][:, :28])
    assert np.array_equal(cho[~ex, 31], (g["moves_len"] > 0).astype(np.int8))
    for i in np.flatnonzero(ex):
        r = pre[i]
        mv, ln, states = orc.turn_sequences(r[:28].astype(np.int32), int(r[28]), int(r[29]), int(r[30]))
        if len(ln) == 0:
            assert np.array_equal(cho[i, :28], r[:28]), i
            continue
        k = (int(x1[i]) * len(ln)) >> 32
        assert np.array_equal(cho[i, :28], states[k].astype(np.int8)) and cho[i, 31] == (ln[k] > 0), i


# ------------------------------------------------------------------ D. long launches: the cache generation wraps

@pytest.mark.gpu
def test_one_cta_select_launch_vs_oracle(fresh, orc, golden, large, defaults):
    """60,000 queries on one CTA of an asynchronous lane: ~3,000 plies per warp, the 8-bit ply generation of every warp's cache
    wraps a dozen times.  The result is the full-grid launch's bit for bit, and the oracle's as in
    test_select_moves_large_sample_vs_oracle."""
    import torch
    w = golden_weights(golden("model.npz"), "trained")
    fresh.set_weights(*w)
    fresh.set_option("select_lane_grid", 1)
    pin = {k: torch.from_numpy(np.zeros_like(defaults["trained", 0.0][k])).pin_memory().numpy() for k in KEYS + ("n_scored",)}
    qp = torch.from_numpy(large.copy()).pin_memory().numpy()
    fresh.select_moves_host_async(0, qp, pin)
    fresh.wait(0)
    assert_same(pin, defaults["trained", 0.0], what="one CTA")
    ref = orc.greedy_batch(w, large)
    assert np.array_equal(pin["n_seq"].astype(np.int64), ref["n_seq"])
    has = ref["n_seq"] > 0
    same = (pin["chosen"][:, :28] == ref["after"]).all(1)
    assert same[~has].all()
    diff = np.flatnonzero(has & ~same)
    for t in (0, 1):
        idx = diff[large[diff, 28] == t]
        if idx.size:
            v = orc.forward(w, orc.encode(pin["chosen"][idx, :28].astype(np.int32), t))
            assert (np.abs(v - ref["value"][idx]) <= 1e-5 * np.abs(ref["value"][idx])).all()
    assert diff.size <= 0.012 * has.sum(), diff.size
    ok = has & same
    assert (np.abs(pin["value"][ok] - ref["value"][ok]) <= 1e-5 * np.abs(ref["value"][ok])).all()
    exact = (pin["moves"].reshape(-1, 8) == ref["moves"].reshape(-1, 8)).all(1) & (pin["moves_len"] == ref["moves_len"])
    assert exact[ok].all()


@pytest.mark.gpu
def test_long_selfplay_step_is_the_host_driven_loop(eng, golden):
    """selfplay_step(600): every warp plays 600 plies of its slot in one launch, more than two wraps of its cache generation."""
    eng.set_weights(*golden_weights(golden("model.npz"), "trained"))
    st = restart_loop_matches_population(eng, 3000, 600)
    assert st["plies"] == 3000 * 600 and st["games_finished"] > 3 * 3000
