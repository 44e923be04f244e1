"""The `*_host` entry points against their device forms: each host form stages its inputs and outputs through engine (or lane)
buffers around the device call, and must give the device call's results bit for bit - with every output, with any one output
alone, across batch sizes that force the staging and work buffers to grow and shrink, at n = 0 and with two lanes in flight.
select_moves' n_scored is the exception: it depends on how the walk was shared between warps, so only its bounds are checked."""
import numpy as np
import pytest
from conftest import golden_weights

pytestmark = pytest.mark.gpu

SEL_ARGS = ("chosen", "moves", "moves_len", "value", "n_seq", "n_scored")     # the outputs of select_moves, in ABI order
SEL_KEYS = SEL_ARGS[:5]                                                        # ... and those that are a function of the query
TWO_KEYS = ("chosen", "moves", "moves_len", "value", "n_candidates", "n_expanded")
ROLL_KEYS = ("mean", "std_err", "counts", "trial_value", "trial_outcome", "trial_plies")


def np_of(x):
    return x.cpu().numpy() if hasattr(x, "cpu") else np.asarray(x)


def same(a, b, what=""):
    a, b = np_of(a), np_of(b)
    assert a.shape == b.shape and a.dtype.itemsize == b.dtype.itemsize, (what, a.shape, b.shape, a.dtype, b.dtype)
    assert np.array_equal(np.ascontiguousarray(a).view(np.uint8), np.ascontiguousarray(b).view(np.uint8)), what


def same_dict(a, b, keys, what=""):
    for k in keys:
        same(a[k], b[k], (what, k))


def check_n_scored(eng, q, out, explore=False):
    """DESIGN 5: every distinct afterstate of a greedy query is scored at least once and nothing beyond its N sequences;
    an explored query scores nothing."""
    U = eng.enumerate_summary_host(q)[1]
    s, N = np_of(out["n_scored"]), np_of(out["n_seq"])
    ok = (s >= U) & (s <= N)
    assert (ok | (s == 0) if explore else ok).all()


def queries(n, seed):
    from bgx.synth import make_queries
    return make_queries(n, seed=seed)[0]


def positions(n, seed):
    q = queries(n, seed).copy()
    q[:, 29:] = 0
    return q


def new_engine(golden):
    from bgx.engine import BatchEngine
    e = BatchEngine(0)
    e.set_weights(*golden_weights(golden("model.npz"), "trained"))
    return e


@pytest.fixture(scope="module")
def eng(golden):
    e = new_engine(golden)
    yield e
    e.close()


def dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def empty(shape, dtype):
    import torch
    return torch.zeros(shape, dtype=dtype, device="cuda:0")


def sel_out(n):
    return {"chosen": np.zeros((n, 32), np.int8), "moves": np.zeros((n, 4, 2), np.int8), "moves_len": np.zeros(n, np.int8),
            "value": np.zeros(n, np.float32), "n_seq": np.zeros(n, np.int32), "n_scored": np.zeros(n, np.int32)}


def two_out(n):
    return {"chosen": np.zeros((n, 32), np.int8), "moves": np.zeros((n, 4, 2), np.int8), "moves_len": np.zeros(n, np.int8),
            "value": np.zeros(n, np.float32), "n_candidates": np.zeros(n, np.int32), "n_expanded": np.zeros(n, np.int32)}


def roll_out(n, trials):
    return {"mean": np.zeros(n, np.float64), "std_err": np.zeros(n, np.float64), "counts": np.zeros((n, 8), np.int64),
            "trial_value": np.zeros((n, trials), np.float32), "trial_outcome": np.zeros((n, trials), np.int8),
            "trial_plies": np.zeros((n, trials), np.int32)}


def raw_select_host(eng, q, o, epsilon=0.0, seed=0):
    from bgx import lib as L
    L.check(eng._lib.bgx_select_moves_host(eng._h, q.ctypes.data, q.shape[0], float(epsilon), int(seed), *(L.ptr(o.get(k)) for k in SEL_ARGS)))


def raw_twoply_host(eng, q, K, o):
    from bgx import lib as L
    L.check(eng._lib.bgx_select_moves_2ply_host(eng._h, q.ctypes.data, q.shape[0], int(K), *(L.ptr(o.get(k)) for k in TWO_KEYS)))


def raw_rollout_host(eng, p, trials, max_plies, o, seed=0x5EED2026, flags=1):
    from bgx import lib as L
    L.check(eng._lib.bgx_rollout_host(eng._h, p.ctypes.data, p.shape[0], int(trials), int(max_plies), int(seed), int(flags),
                                      *(L.ptr(o.get(k)) for k in ROLL_KEYS)))


# ------------------------------------------------------------------ host form == device form

def test_host_forms_equal_device_forms(eng):
    import torch
    q = queries(3000, seed=11)
    n = len(q)
    dq = dev(q)

    X = empty((n, 198), torch.float32)
    eng.encode(dq, X)
    V = empty(n, torch.float32)
    eng.evaluate(dq, V)
    ns, nu, dg = empty(n, torch.int32), empty(n, torch.int32), empty(n, torch.int64)
    eng.enumerate_summary(dq, ns, nu, dg)
    cnt, off = empty(n, torch.int32), empty(n + 1, torch.int64)
    eng.enumerate_count(dq, cnt, off)
    eng.synchronize()
    rows = int(off[-1])
    mv, ln, st = empty((rows, 4, 2), torch.int8), empty(rows, torch.int8), empty((rows, 32), torch.int8)
    eng.enumerate(dq, off, mv, ln, st)
    d_sel = {k: empty(a.shape, getattr(torch, str(a.dtype))) for k, a in sel_out(n).items()}
    eng.select_moves(dq, 0.0, 0, **d_sel)
    d_sel_x = {k: empty(a.shape, getattr(torch, str(a.dtype))) for k, a in sel_out(n).items()}
    eng.select_moves(dq, 0.25, 77, **d_sel_x)
    eng.synchronize()

    same(eng.encode_host(q), X, "encode")
    same(eng.evaluate_host(q), V, "evaluate")
    h_ns, h_nu, h_dg = eng.enumerate_summary_host(q)
    same(h_ns, ns, "n_seq"); same(h_nu, nu, "n_unique"); same(h_dg, dg, "digest")
    h_off, h_mv, h_ln, h_st = eng.enumerate_host(q)
    same(h_off, off, "offsets"); same(h_mv, mv, "moves"); same(h_ln, ln, "lens"); same(h_st, st, "states")
    same(cnt, h_ns, "enumerate_count n_seq")
    for eps, seed, d in ((0.0, 0, d_sel), (0.25, 77, d_sel_x)):
        h = eng.select_moves_host(q, eps, seed)
        same_dict(h, d, SEL_KEYS, ("select", eps))
        check_n_scored(eng, q, h, eps > 0)
        check_n_scored(eng, q, d, eps > 0)

    q2 = q[:300]
    for K in (0, 3):
        d_two = {k: empty(a.shape, getattr(torch, str(a.dtype))) for k, a in two_out(len(q2)).items()}
        eng.select_moves_2ply(dev(q2), K, **d_two)
        eng.synchronize()
        same_dict(eng.select_moves_2ply_host(q2, K), d_two, TWO_KEYS, ("2ply", K))

    p = positions(12, seed=5)
    for max_plies, stratify in ((0, True), (9, False)):
        d_roll = eng.rollout(dev(p), 72, max_plies=max_plies, stratify=stratify, per_trial=True)
        eng.synchronize()
        same_dict(eng.rollout_host(p, 72, max_plies=max_plies, stratify=stratify, per_trial=True), d_roll, ROLL_KEYS, ("rollout", max_plies))

    eng.selfplay_init(64, traj_cap=256)
    eng.selfplay_step(40)
    out = empty((64 * 5, 32), torch.int8)
    eng.selfplay_sample(5, 123, out)
    eng.synchronize()
    same(eng.selfplay_sample_host(5, 123), out, "selfplay_sample")


# ------------------------------------------------------------------ one optional output at a time

def test_single_outputs_equal_all_outputs(eng):
    import torch
    q = queries(2000, seed=21)
    n = len(q)
    full = sel_out(n)
    raw_select_host(eng, q, full, 0.1, 9)
    for k in SEL_ARGS:
        one = {k: np.zeros_like(full[k])}
        raw_select_host(eng, q, one, 0.1, 9)
        pin = {k: torch.from_numpy(np.zeros_like(full[k])).pin_memory().numpy()}
        eng.select_moves_host_async(1, q, pin, epsilon=0.1, seed=9)
        eng.wait(1)
        for o, what in ((one, "select_moves_host"), (pin, "select_moves_host_async")):
            if k == "n_scored":
                check_n_scored(eng, q, {"n_scored": o[k], "n_seq": full["n_seq"]}, explore=True)
            else:
                same(o[k], full[k], (what, k))

    q2 = q[:200]
    full = two_out(len(q2))
    raw_twoply_host(eng, q2, 2, full)
    for k in TWO_KEYS:
        one = {k: np.zeros_like(full[k])}
        raw_twoply_host(eng, q2, 2, one)
        same(one[k], full[k], ("select_moves_2ply_host", k))

    p = positions(6, seed=8)
    full = roll_out(len(p), 36)
    raw_rollout_host(eng, p, 36, 0, full)
    for k in ROLL_KEYS:
        one = {k: np.zeros_like(full[k])}
        raw_rollout_host(eng, p, 36, 0, one)
        same(one[k], full[k], ("rollout_host", k))
    for per_trial in (False, True):
        o = eng.rollout_host(p, 36, per_trial=per_trial)
        same_dict(o, full, ROLL_KEYS if per_trial else ROLL_KEYS[:3], ("rollout_host per_trial", per_trial))


# ------------------------------------------------------------------ staging and work buffers grow and shrink mid-sequence

def test_interleaved_sizes_equal_fresh_engine(eng, golden):
    calls = []
    for n in (37, 12000, 50, 9000, 3):
        q = queries(n, seed=1000 + n)
        calls += [
            ("encode", q, lambda e, q=q: e.encode_host(q)),
            ("select", q, lambda e, q=q: e.select_moves_host(q)),
            ("summary", q, lambda e, q=q: e.enumerate_summary_host(q)),
            ("evaluate", q, lambda e, q=q: e.evaluate_host(q)),
            ("enumerate", q, lambda e, q=q: e.enumerate_host(q)),
            ("2ply", q, lambda e, q=q: e.select_moves_2ply_host(q[:max(1, len(q) // 20)], 2)),
            ("rollout", q, lambda e, q=q: e.rollout_host(positions(max(1, len(q) // 1000), seed=len(q)), 36, max_plies=30, per_trial=True)),
        ]
    got = [f(eng) for _, _, f in calls]
    for (name, q, f), g in zip(calls, got):
        ref = new_engine(golden)
        try:
            r = f(ref)
        finally:
            ref.close()
        if name == "select":
            check_n_scored(eng, q, g)
            g, r = ({k: d[k] for k in SEL_KEYS} for d in (g, r))
        pairs = zip(g.values(), r.values()) if isinstance(g, dict) else zip(g, r) if isinstance(g, tuple) else [(g, r)]
        for a, b in pairs:
            same(a, b, name)


# ------------------------------------------------------------------ n = 0

def test_empty_batches(eng):
    z = np.zeros((0, 32), np.int8)
    assert eng.encode_host(z).shape == (0, 198)
    assert eng.evaluate_host(z).shape == (0,)
    assert all(a.shape == (0,) for a in eng.enumerate_summary_host(z))
    off, mv, _, _ = eng.enumerate_host(z)
    assert off.tolist() == [0] and mv.shape[0] == 0
    assert eng.select_moves_host(z)["chosen"].shape == (0, 32)
    assert eng.select_moves_2ply_host(z, 0)["chosen"].shape == (0, 32)
    assert eng.rollout_host(z, 36, per_trial=True)["mean"].shape == (0,)
    eng.select_moves_host_async(0, z, sel_out(0))
    eng.wait(0)
    e32, e64 = np.zeros(0, np.int32), np.zeros(0, np.int64)
    eng.play_ply_host_async(1, z, e32, e64, np.zeros((0, 32), np.int8))
    eng.wait(1)
    eng.play_ply_restart_host_async(2, z, e32, e64, 1, np.zeros((0, 32), np.int8))
    eng.wait(2)
    # the lanes still work after an empty batch
    q = queries(100, seed=3)
    o = sel_out(100)
    eng.select_moves_host_async(0, q, o)
    eng.wait(0)
    same_dict(o, eng.select_moves_host(q), SEL_KEYS, "after n = 0")
    check_n_scored(eng, q, o)


# ------------------------------------------------------------------ lanes in flight together

def test_two_lanes_in_flight_equal_synchronous_calls(eng):
    import torch
    from bgx import host as H
    qa, qb = queries(7000, seed=31), queries(5000, seed=32)
    want_a, want_b = eng.select_moves_host(qa), eng.select_moves_host(qb, 0.2, 5)
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()
    oa = {k: pin(np.zeros_like(v)) for k, v in want_a.items()}
    ob = {k: pin(np.zeros_like(v)) for k, v in want_b.items()}
    eng.select_moves_host_async(0, pin(qa), oa)
    eng.select_moves_host_async(1, pin(qb), ob, epsilon=0.2, seed=5)
    eng.wait(1)
    eng.wait(0)
    same_dict(oa, want_a, SEL_KEYS, "lane 0")
    same_dict(ob, want_b, SEL_KEYS, "lane 1")
    check_n_scored(eng, qa, oa)
    check_n_scored(eng, qb, ob, explore=True)

    # two play-ply batches in flight, twice over, so that the second call of each lane reads the queue the first left
    rng = np.random.default_rng(4)
    batches = []
    for q in (qa, qb):
        n = len(q)
        ply, gid = rng.integers(0, 300, n).astype(np.int32), rng.integers(0, 2 ** 40, n).astype(np.int64)
        ref = eng.select_moves_host(q)
        nxt, win = np.zeros((n, 32), np.int8), np.zeros(n, np.int8)
        H.advance(ref["chosen"], nxt, 99, ply, gid, win)
        batches.append((pin(q), pin(ply), pin(gid), ref, nxt, win))
    for _ in range(2):
        outs = []
        for lane, (q, ply, gid, _, _, _) in zip((2, 3), batches):
            n = len(q)
            o = (pin(np.zeros((n, 32), np.int8)), pin(np.full(n, 9, np.int8)), pin(np.zeros(n, np.float32)), pin(np.zeros(n, np.int32)))
            eng.play_ply_host_async(lane, q, ply, gid, *o, dice_seed=99)
            outs.append(o)
        eng.wait(2)
        eng.wait(3)
        for (_, _, _, ref, nxt, win), (g_nxt, g_win, g_val, g_nseq) in zip(batches, outs):
            same(g_nxt, nxt, "next records")
            same(g_win, win, "winner")
            same(g_nseq, ref["n_seq"], "n_seq")
            ok = ref["n_seq"] > 0
            same(g_val[ok], ref["value"][ok], "value")
