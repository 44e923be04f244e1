"""Variance-reduced rollouts (DESIGN 7e, bgx_rollout_vr): the restatement against rollout_ref and its own identities on the CPU; on
the GPU the fused kernel against the host-driven loop over the one-ply kernel (bit for bit), against bgx_rollout's play, against
two-ply's expectation at T = 1, against the CPU oracle under exact tie nets, as a pure function of its inputs, on its edge cases,
statistically against the plain estimate and through every surface."""
import numpy as np
import pytest
from conftest import golden_weights
from rollout_ref import MAX_PLIES, engine_ply, oracle_ply, reduce_trials, rollout
from rollout_vr_ref import rollout_vr
from test_ply_exactness import tie_net
from test_rollout import SEED, START, OUT_KEYS, board, positions, rec_of, same, weights_of

VR_KEYS = ("vr_mean", "vr_std_err", "trial_luck")


def luck_upto(ref, events, vr):
    """ref (a rollout_vr result at vr_plies >= every trial's plies) re-reduced for vr_plies = vr from its per-ply luck events"""
    n, T = ref["trial_value"].shape
    luck = np.zeros(n * T)
    for items, ply, _, _, lk in events:
        m = ply < vr
        luck[items[m]] = luck[items[m]] + lk[m]
    out = dict(ref)
    out["trial_luck"] = luck.reshape(n, T)
    out["vr_mean"], out["vr_std_err"] = np.zeros(n), np.zeros(n)
    for p in range(n):
        y = ref["trial_value"][p].astype(np.float64) - out["trial_luck"][p]
        out["vr_mean"][p], out["vr_std_err"][p], _ = reduce_trials(y, ref["trial_outcome"][p], ref["trial_plies"][p])
    return out


def recorded(ply_fn, value_fn, pos, trials, **kw):
    events = []
    ref = rollout_vr(ply_fn, value_fn, pos, trials, vr_plies=MAX_PLIES, on_vr_ply=lambda *a: events.append(a), **kw)
    return ref, events


# ------------------------------------------------------------------ CPU

@pytest.mark.parametrize("kind", ("off", "bar"))
def test_restatement_without_vr_is_the_rollout(orc, kind):
    """vr_plies = 0: the restatement is rollout_ref.rollout bit for bit, luck 0 and vr_mean = mean."""
    ply, value = oracle_ply(orc, tie_net(kind))
    pos = positions(4, seed=4242)
    for T, strat in ((0 if kind == "off" else 24, True), (7, False)):
        got = rollout_vr(ply, value, pos, 36, max_plies=T, vr_plies=0, stratify=strat)
        same(got, rollout(ply, value, pos, 36, max_plies=T, stratify=strat), what=(kind, T))
        assert (got["trial_luck"] == 0).all()
        same({"vr_mean": got["vr_mean"], "vr_std_err": got["vr_std_err"]}, {"vr_mean": got["mean"], "vr_std_err": got["std_err"]},
             keys=("vr_mean", "vr_std_err"))


@pytest.mark.parametrize("kind", ("off", "bar"))
def test_first_roll_luck_sums_to_zero(orc, kind):
    """36 stratified trials play each ordered first roll once: their ply-0 luck sums to 0 within float64 rounding, and at T = 1 each
    y_t of a trial that did not end the game is E_0 within a few ulps."""
    ply, value = oracle_ply(orc, tie_net(kind))
    pos = positions(6, seed=515)
    events = []
    out = rollout_vr(ply, value, pos, 36, max_plies=1, vr_plies=1, stratify=True, on_vr_ply=lambda *a: events.append(a))
    (items, plies, L, E, lk), = events
    assert (plies == 0).all() and len(items) == len(pos) * 36
    for p in range(len(pos)):
        assert abs(sum(out["trial_luck"][p].tolist())) <= 1e-13, (kind, p)
        E0 = E[items // 36 == p]
        assert np.all(E0 == E0[0])
        y = out["trial_value"][p].astype(np.float64) - out["trial_luck"][p]
        live = out["trial_outcome"][p] == 0
        assert live.any()
        assert np.all(np.abs(y[live] - E0[0]) <= 4 * np.finfo(np.float64).eps * max(1.0, abs(E0[0]))), (kind, p)


# ------------------------------------------------------------------ GPU

@pytest.fixture(scope="module")
def eng():
    from bgx.engine import BatchEngine
    e = BatchEngine(0)
    yield e
    e.close()


def vr_host(eng, pos, trials, vr, max_plies=0, seed=SEED, stratify=True):
    """bgx_rollout_vr_host through ctypes, every output (vr = 0 included, which BatchEngine routes to bgx_rollout)"""
    from bgx import lib as L
    n = len(pos)
    o = {"mean": np.zeros(n), "std_err": np.zeros(n), "counts": np.zeros((n, 8), np.int64),
         "trial_value": np.zeros((n, trials), np.float32), "trial_outcome": np.zeros((n, trials), np.int8),
         "trial_plies": np.zeros((n, trials), np.int32), "vr_mean": np.zeros(n), "vr_std_err": np.zeros(n),
         "trial_luck": np.zeros((n, trials))}
    q = np.ascontiguousarray(pos, np.int8)
    L.check(eng._lib.bgx_rollout_vr_host(eng._h, q.ctypes.data, n, trials, max_plies, seed, L.ROLLOUT_STRATIFY if stratify else 0, vr,
                                         *eng._rollout_outputs(o)))
    return o


@pytest.mark.gpu
@pytest.mark.parametrize("net", ("trained", "rand"))
def test_rollout_vr_is_the_host_driven_loop(eng, golden, net):
    """256 positions x 72 trials, T in {0, 1, 2, 7}, vr_plies in {1, 3, 4096}, stratified and not: trial_luck, vr_mean and
    vr_std_err equal the restatement over select_moves_host / evaluate_host bit for bit, and the play and bgx_rollout's outputs
    equal bgx_rollout's."""
    eng.set_weights(*weights_of(golden, net))
    pos = positions(256, seed=31337)
    ply, value = engine_ply(eng)
    for T in (0, 1, 2, 7):
        for strat in (True, False):
            ref, events = recorded(ply, value, pos, 72, max_plies=T, seed=SEED, stratify=strat)
            plain = eng.rollout_host(pos, 72, max_plies=T, seed=SEED, stratify=strat, per_trial=True)
            same(plain, ref, what=(net, T, strat, "plain"))
            for vr in (1, 3, MAX_PLIES):
                got = eng.rollout_host(pos, 72, max_plies=T, seed=SEED, stratify=strat, per_trial=True, vr_plies=vr)
                same(got, plain, what=(net, T, strat, vr, "play"))
                same(got, luck_upto(ref, events, vr), keys=VR_KEYS, what=(net, T, strat, vr))
            assert (got["trial_luck"] != 0).any()


@pytest.mark.gpu
def test_vr_plies_zero_is_the_plain_rollout(eng, golden):
    """bgx_rollout_vr at vr_plies = 0: every output of bgx_rollout, luck exactly 0, vr_mean = mean, vr_std_err = std_err."""
    eng.set_weights(*golden_weights(golden("model.npz"), "trained"))
    pos = positions(32, seed=808)
    for T in (0, 5):
        got = vr_host(eng, pos, 72, 0, max_plies=T)
        same(got, eng.rollout_host(pos, 72, max_plies=T, seed=SEED, per_trial=True), what=T)
        assert (got["trial_luck"] == 0).all()
        same({"vr_mean": got["mean"], "vr_std_err": got["std_err"]}, got, keys=("vr_mean", "vr_std_err"))


@pytest.mark.gpu
def test_one_ply_vr_rollout_is_twoply_expectation(eng, golden):
    """Two-ply's pick A with the opponent on roll, T = 1, vr_plies = 1, where no reply can win (the opponent has <= 10 borne off):
    every y_t is E_0, so vr_mean is two-ply's value within one fp32 ulp and vr_std_err <= 1e-12; and float32(E_0) of the restatement
    is two-ply's value bit for bit (the same float64 sum, rounded once)."""
    from bgx.synth import make_queries
    eng.set_weights(*golden_weights(golden("model.npz"), "trained"))
    q = make_queries(512, seed=2468)[0]
    two = eng.select_moves_2ply_host(q, max_candidates=0)
    A = two["chosen"].copy()
    p = q[:, 28].astype(np.int64)
    usable = (two["n_candidates"] > 0) & (A[:, 26] != 15) & (A[:, 27] != 15)
    A[:, 28] = 1 - p
    A[:, 29:] = 0
    no_win = A[np.arange(len(A)), 26 + A[:, 28].astype(np.int64)] <= 10
    keep = usable & no_win
    A = A[keep]
    v2 = two["value"][keep]
    assert len(A) > 300
    ro = eng.rollout_host(A, 36, max_plies=1, seed=SEED, stratify=True, per_trial=True, vr_plies=1)
    assert (ro["trial_plies"] == 1).all() and (ro["trial_outcome"] == 0).all()
    ulp = np.spacing(np.abs(v2)).astype(np.float64)
    assert np.all(np.abs(ro["vr_mean"] - v2.astype(np.float64)) <= ulp)
    assert (ro["vr_std_err"] <= 1e-12).all()
    E0 = {}
    rollout_vr(*engine_ply(eng), A, 36, max_plies=1, vr_plies=1, seed=SEED,
               on_vr_ply=lambda items, ply, L, E, lk: E0.update(zip((items // 36).tolist(), E.tolist())))
    E0 = np.array([E0[i] for i in range(len(A))])
    assert np.array_equal(E0.astype(np.float32).view(np.uint32), v2.view(np.uint32))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ("off", "bar"))
def test_rollout_vr_tie_nets_are_the_oracle(eng, orc, kind):
    """Under an exact tie net: 8 positions x 72 trials against the CPU oracle's restatement.  Outcomes, plies and counts are equal;
    the luck, a sum of differences of sigmoids (expf in the oracle, the SFU in the kernel), agrees to 2e-6 per value."""
    w = tie_net(kind)
    eng.set_weights(*w)
    pos = positions(8, seed=777)
    for T, vr, strat in ((0 if kind == "off" else 48, 3, True), (7, MAX_PLIES, False)):
        got = eng.rollout_host(pos, 72, max_plies=T, seed=SEED, stratify=strat, per_trial=True, vr_plies=vr)
        want = rollout_vr(*oracle_ply(orc, w), pos, 72, max_plies=T, vr_plies=vr, seed=SEED, stratify=strat)
        same(got, want, keys=("trial_outcome", "trial_plies", "counts"), what=(kind, T))
        k = np.minimum(got["trial_plies"], vr)
        assert np.all(np.abs(got["trial_luck"] - want["trial_luck"]) <= 4e-6 * np.maximum(k, 1)), kind
        assert (got["trial_luck"] != 0).any()


@pytest.mark.gpu
def test_rollout_vr_is_a_pure_function(eng, golden):
    """The same positions give bit-identical outputs alone, inside a larger batch permuted and duplicated, under every chunking and
    every warps-per-CTA setting."""
    eng.set_weights(*golden_weights(golden("model.npz"), "trained"))
    pos = positions(24, seed=99)
    kw = dict(seed=SEED, per_trial=True, vr_plies=3)
    keys = OUT_KEYS + VR_KEYS
    base = eng.rollout_host(pos, 72, **kw)
    other = positions(40, seed=100)
    big = np.concatenate([pos, other, pos[:8]])
    perm = np.random.default_rng(5).permutation(len(big))
    got = eng.rollout_host(big[perm], 72, **kw)
    inv = np.argsort(perm)
    same({k: v[inv[:24]] for k, v in got.items()}, base, keys=keys, what="batch")
    same({k: v[inv[64:72]] for k, v in got.items()}, {k: v[:8] for k, v in base.items()}, keys=keys, what="duplicates")
    for chunk in (72, 7 * 72, 0):
        eng.set_option("rollout_chunk", chunk)
        same(eng.rollout_host(pos, 72, **kw), base, keys=keys, what=("chunk", chunk))
    eng.set_option("rollout_chunk", 0)
    for warps in (16, 24, 32, 20):
        eng.set_option("rollout_warps", warps)
        same(eng.rollout_host(pos, 72, **kw), base, keys=keys, what=("warps", warps))
    # without the per-trial arrays: the same outputs (per-trial results in engine scratch)
    same(eng.rollout_host(pos, 72, seed=SEED, vr_plies=3), base, keys=("mean", "std_err", "counts", "vr_mean", "vr_std_err"),
         what="scratch")


@pytest.mark.gpu
def test_rollout_vr_edges(eng, golden):
    from bgx import lib as L
    eng.set_weights(*golden_weights(golden("model.npz"), "trained"))
    ply, value = engine_ply(eng)
    # finished positions: no ply, no luck
    done = np.stack([rec_of(board(p1=-14, p19=-1), off=(15, 0), player=1), rec_of(board(p24=12), off=(3, 15), player=0)])
    o = eng.rollout_host(done, 36, seed=SEED, per_trial=True, vr_plies=MAX_PLIES)
    assert (o["trial_luck"] == 0).all() and list(o["vr_mean"]) == [1.0, 0.0] and list(o["vr_std_err"]) == [0.0, 0.0]
    # every roll blocked at ply 0 (PLAYER2 on the bar against a closed board): L = V for all 21 rolls, luck exactly 0 there
    closed = board(p19=2, p20=2, p21=2, p22=2, p23=2, p24=2, p11=3, p1=-4, p2=-4, p3=-3, p4=-3)
    blocked = np.stack([rec_of(closed, bar=(0, 1), player=1)] * 2)
    got = eng.rollout_host(blocked, 36, max_plies=1, seed=SEED, per_trial=True, vr_plies=1)
    assert (got["trial_luck"] == 0).all() and (got["vr_mean"] == got["mean"]).all()
    ref, events = recorded(ply, value, blocked, 36, max_plies=9, seed=SEED)
    assert (events[0][4] == 0).all()
    got = eng.rollout_host(blocked, 36, max_plies=9, seed=SEED, per_trial=True, vr_plies=MAX_PLIES)
    same(got, ref, keys=OUT_KEYS + VR_KEYS, what="blocked")
    # vr_plies beyond every trial: the same as vr_plies = the cut
    pos = positions(16, seed=12)
    a = eng.rollout_host(pos, 36, max_plies=7, seed=SEED, per_trial=True, vr_plies=MAX_PLIES)
    same(a, eng.rollout_host(pos, 36, max_plies=7, seed=SEED, per_trial=True, vr_plies=7), keys=OUT_KEYS + VR_KEYS, what="beyond")
    # no positions, both forms
    o = eng.rollout_host(np.zeros((0, 32), np.int8), 36, per_trial=True, vr_plies=2)
    assert o["vr_mean"].shape == (0,) and o["trial_luck"].shape == (0, 36)
    import torch
    o = eng.rollout(torch.zeros((0, 32), dtype=torch.int8, device="cuda"), 36, per_trial=True, vr_plies=2)
    assert tuple(o["vr_mean"].shape) == (0,) and tuple(o["trial_luck"].shape) == (0, 36)
    # invalid arguments: bgx_rollout's, and vr_plies outside [0, BGX_ROLLOUT_MAX_PLIES]
    for kw in ({"trials": 35}, {"trials": 72, "max_plies": -1}, {"trials": 72, "vr_plies": -1}, {"trials": 72, "vr_plies": MAX_PLIES + 1}):
        with pytest.raises(L.BgxError) as ei:
            eng.rollout_host(pos[:2], **{"vr_plies": 1, **kw})
        assert ei.value.code == L.E_INVALID
    q = np.ascontiguousarray(pos[:2])
    for vr in (-1, MAX_PLIES + 1):
        assert eng._lib.bgx_rollout_vr(eng._h, q.ctypes.data, 2, 36, 0, SEED, 1, vr, *([None] * 9)) == L.E_INVALID


@pytest.mark.gpu
def test_long_vr_trials_under_the_bar_net(eng):
    """Under the bar net trials run to hundreds of plies; cut at 300 with VR on every ply: still the host-driven loop bit for bit."""
    eng.set_weights(*tie_net("bar"))
    pos = positions(6, seed=4242)[4:]
    got = eng.rollout_host(pos, 36, max_plies=300, seed=SEED, per_trial=True, vr_plies=MAX_PLIES)
    want = rollout_vr(*engine_ply(eng), pos, 36, max_plies=300, vr_plies=MAX_PLIES, seed=SEED)
    same(got, want, keys=OUT_KEYS + VR_KEYS, what="bar")
    assert np.median(got["trial_plies"]) > 200


@pytest.mark.gpu
def test_vr_statistics(eng, golden):
    """The opening (each side on roll) and 14 self-play positions, 12,960 stratified trials, VR on every ply: vr_mean and mean agree
    within 4 combined sigma, and VR lowers the standard error (median vr_std_err / std_err below 1; measured on an NVIDIA B200 at
    1,000 W: 0.65, per position 0.57 .. 1.07).  A sampled position that is
    already decided has no variance to reduce and is left out of the ratio."""
    from bgx.lib import FIRST_PARITY
    eng.set_weights(*golden_weights(golden("model.npz"), "trained"))
    eng.selfplay_init(14, first_id=0, id_stride=14, seed=20261022, first_mover=FIRST_PARITY, traj_cap=1024)
    eng.selfplay_round()
    sp = eng.selfplay_sample_host(1, seed=20261022)
    sp[:, 29:] = 0
    pos = np.concatenate([np.stack([rec_of(START, player=0), rec_of(START, player=1)]), sp])
    o = eng.rollout_host(pos, 12960, seed=SEED, vr_plies=MAX_PLIES)
    sigma = np.sqrt(o["std_err"] ** 2 + o["vr_std_err"] ** 2)
    assert np.all(np.abs(o["vr_mean"] - o["mean"]) <= 4 * sigma), (o["vr_mean"], o["mean"], sigma)
    live = o["std_err"] > 0
    assert live[:2].all() and live.sum() >= 12
    ratio = o["vr_std_err"][live] / o["std_err"][live]
    print("vr_std_err / std_err per position:", np.round(ratio, 3).tolist(), "median", float(np.median(ratio)))
    assert np.median(ratio) < 1


@pytest.mark.gpu
def test_rollout_vr_surfaces_agree(eng, golden):
    """ctypes host and device forms, the pybind module and TDLGammonModel.rollout_batch give the same results bit for bit."""
    import torch
    import backgammon_env as bg
    from bgx.model import TDLGammonModel
    w = golden_weights(golden("model.npz"), "trained")
    eng.set_weights(*w)
    pos = positions(16, seed=55)
    host = eng.rollout_host(pos, 72, max_plies=0, seed=SEED, per_trial=True, vr_plies=4)
    dev = eng.rollout(torch.from_numpy(pos).cuda(), 72, max_plies=0, seed=SEED, per_trial=True, vr_plies=4)
    torch.cuda.synchronize()
    same(host, {k: v.cpu().numpy() for k, v in dev.items()}, keys=OUT_KEYS + VR_KEYS, what="device")
    pb = bg.BatchEngine(0)
    pb.set_weights(*w)
    same(host, pb.rollout(pos, 72, 0, SEED, True, True, 4), keys=OUT_KEYS + VR_KEYS, what="pybind")
    same(host, vr_host(eng, pos, 72, 4), keys=OUT_KEYS + VR_KEYS, what="ctypes")
    m = TDLGammonModel()
    W1, b1, w2, b2 = w
    m.load_state_dict({"fc1.weight": torch.from_numpy(W1), "fc1.bias": torch.from_numpy(b1),
                       "fc2.weight": torch.from_numpy(w2), "fc2.bias": torch.from_numpy(b2)})
    free = pos[(pos[:, 24] == 0) & (pos[:, 25] == 0)]               # the compat Game has no setter for the bar
    games = []
    for r in free:
        g = bg.Game(0)
        g.setGameBoard([int(x) for x in r[:24]])
        g.setBorneOffPieces(0, int(r[26]))
        g.setBorneOffPieces(1, int(r[27]))
        g.setTurn(int(r[28]))
        g.roll_dice()
        games.append(g)
    want = eng.rollout_host(free, 72, seed=SEED, vr_plies=4)
    rb = m.rollout_batch(games, trials=72, seed=SEED, vr_plies=4)
    assert np.array_equal(rb["p1_win"], want["mean"]) and np.array_equal(rb["vr_p1_win"], want["vr_mean"])
    assert np.array_equal(rb["vr_std_err"], want["vr_std_err"])
