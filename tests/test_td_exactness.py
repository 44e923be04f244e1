"""k_td_replay (bgx_td.cuh) the way training runs it, where the rest of the suite has slack or does not reach:
  A. a population replay, several games per CTA, equals the per-game replays bit for bit: within one game nothing depends on
     the CTA or on what it replayed before (its home tables start every game as the snapshot), so every game's final weights
     are bgx_td_replay_host's, and the round delta is a fixed fp32 sum of them (DESIGN §3) that numpy reproduces exactly.
     The replay's counters are exact too;
  B. single games at the edges (T = 1 .. 18 around the record ring and the 4-step lazy trips, T = 2048 = kTdMaxSteps, lambda 0
     and 1, lr 1), against torch and float64, per tensor and per feature row, and lr = 0 exactly;
  C. the kernel's own feature values (TdLaneRow, the class colouring, the borne-off table) over their whole domain, through
     the values it computes at lr = 0, state by state."""
import numpy as np
import pytest

from conftest import golden_weights
from test_ply_exactness import tie_net

SEED = 0x5EED2026
LR, LAM = 0.1, 0.9
NPARAMS, NPARAMS_PADDED = 25601, 25604
BOUNDS = (0, 25344, 25472, 25600, 25601)
TENSORS = ("W1", "b1", "w2", "b2")
TD_CTAS_PER_SM = 4                       # kTdCtasPerSm (bgx_td.cuh): the replay's grid is min(4 x SMs, games)
TD_MAX_STEPS = 2048                      # kTdMaxSteps
P1_WON, P2_WON, TRUNCATED = 1, 2, 3      # byte 31 of a slot
CAP = 56                                 # the small trajectory cap of the truncating population


def flat(weights):
    return np.concatenate([np.asarray(a, np.float32).reshape(-1) for a in weights])


def encode(orc, rec):
    """records int8[T, 32] (byte 28 = turn flag) -> the model's features float32[T, 198] (orc_encode)"""
    rec = np.asarray(rec)
    X = np.zeros((len(rec), 198), np.float32)
    for turn in (0, 1):
        m = (rec[:, 28] != 0) == bool(turn)
        if m.any():
            X[m] = orc.encode(rec[m, :28].astype(np.int32), turn)
    return X


def forward64(w, X):
    W1, b1, w2, b2 = (np.asarray(a, np.float64) for a in w)
    h = 1.0 / (1.0 + np.exp(-(np.asarray(X, np.float64) @ W1.reshape(128, 198).T + b1)))
    return 1.0 / (1.0 + np.exp(-(h @ w2.reshape(-1) + b2.reshape(-1)[0])))


def same_bits(a, b):
    a, b = np.ascontiguousarray(a, np.float32), np.ascontiguousarray(b, np.float32)
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


# ------------------------------------------------------------------ A. the round delta, emulated on the host

def emulate_round_delta(finals, n_slots, grid, w0):
    """The exact fp32 delta of bgx_td_replay from the final weights of every finished game.
    finals: (slot, flat final weights float32[25601]) of the won slots in ascending slot order; every other slot contributes
    nothing.  CTA b replays slots b, b + grid, ... (grid = min(kTdCtasPerSm x SMs, n_slots)) and adds fp32(w_final - w0)
    to its accumulator in that order; k_td_reduce then sums the accumulators over CTAs 0 .. grid-1, one fp32 add at a time.
    A row a game never touched adds w0 - w0 = +0, which leaves an accumulator as it is."""
    w0 = flat(w0)
    acc = np.zeros((grid, NPARAMS_PADDED), np.float32)
    for slot, new in finals:
        assert 0 <= slot < n_slots
        acc[slot % grid, :NPARAMS] += np.asarray(new, np.float32) - w0
    delta = np.zeros(NPARAMS_PADDED, np.float32)
    for c in range(grid):
        delta += acc[c]
    delta[NPARAMS:] = 0.0
    return delta


def replay_counts(X):
    """-> (live row-steps, lazily replayed row-steps) of one game, as k_td_replay counts them: a row is live at step t when
    its feature is non-zero in s_t, s_t+1 or s_t+2 (0 beyond the game); a touched row replays lazily every step from its
    first live step on that it was not live at."""
    T = len(X)
    nz = np.zeros((T + 2, 198), bool)
    nz[:T] = X != 0
    live = nz[:T] | nz[1:T + 1] | nz[2:T + 2]
    n_live = live.sum(0)
    touched = n_live > 0
    first = np.argmax(live, 0)
    return int(n_live.sum()), int((T - first - n_live)[touched].sum())


class Population:
    """A self-play round of n_slots games from the current weights, read back with every slot's trajectory."""

    def __init__(self, eng, n_slots, traj_cap, seed=SEED, play=True):
        self.n, self.cap = n_slots, traj_cap
        eng.selfplay_init(n_slots, first_id=0, id_stride=n_slots, seed=seed, traj_cap=traj_cap)
        if play:
            eng.selfplay_round()
            self.read(eng)

    def read(self, eng):
        rec, self.ply, _ = eng.selfplay_read()
        self.status = rec[:, 31].copy()
        self.won = (self.status == P1_WON) | (self.status == P2_WON)
        self.trajs = [eng.export_trajectory(s)[0] if self.won[s] else None for s in range(self.n)]


def check_round(eng, orc, pop, delta, st, params):
    """bgx_td_replay's delta and counters (delta: the device tensor it wrote, st: its stats) against the emulated round built
    from bgx_td_replay_host on every finished game with the engine's current weights; params(slot) -> (lr, lambda)."""
    import torch
    torch.cuda.synchronize()
    got = delta.cpu().numpy()
    w0 = eng.get_weights()
    grid = min(TD_CTAS_PER_SM * eng.device_props()["sm_count"], pop.n)
    slots = np.flatnonzero(pop.won)
    X_all = encode(orc, np.concatenate([pop.trajs[s] for s in slots]))
    want = {"td_steps": 0, "games_finished": len(slots), "truncated": int((pop.status == TRUNCATED).sum()),
            "td_live_rows": 0, "td_lazy_row_steps": 0}
    sq_total = 0.0

    def finals():
        nonlocal sq_total
        at = 0
        for s in slots:
            rec = pop.trajs[s]
            T = len(rec)
            assert T == min(pop.ply[s], pop.cap, TD_MAX_STEPS) and T > 0
            new, sq = eng.td_replay_host(rec, pop.status[s] == P1_WON, *params(s))
            sq_total += float(sq.sum())
            live, lazy = replay_counts(X_all[at:at + T])
            at += T
            want["td_steps"] += T
            want["td_live_rows"] += live
            want["td_lazy_row_steps"] += lazy
            yield s, flat(new)
    emulated = emulate_round_delta(finals(), pop.n, grid, w0)
    assert same_bits(eng.get_weights()[0], w0[0])                       # the single-game replays left the snapshot alone
    bad = np.flatnonzero(got.view(np.uint32) != emulated.view(np.uint32))
    assert len(bad) == 0, ("delta differs from the emulated round", len(bad), bad[:8].tolist(),
                           float(np.max(np.abs(got.astype(np.float64) - emulated))))
    for k, v in want.items():
        assert st[k] == v, (k, st[k], v)
    # the float64 sum of squared TD errors is an atomicAdd across CTAs: its order is not fixed
    assert abs(st["td_sq_error"] - sq_total) <= 1e-12 * sq_total, (st["td_sq_error"], sq_total)
    return grid


@pytest.fixture(scope="module")
def eng():
    from bgx.engine import BatchEngine
    e = BatchEngine(0)
    yield e
    e.close()


def population_size(eng):
    """Not a multiple of the replay's grid, with six or seven games on every CTA (4,099 on a 148-SM B200)."""
    grid = TD_CTAS_PER_SM * eng.device_props()["sm_count"]
    return 7 * grid - 45


def new_delta():
    import torch
    return torch.full((NPARAMS_PADDED,), float("nan"), device="cuda", dtype=torch.float32)


@pytest.mark.gpu
@pytest.mark.parametrize("net,cap", [("trained", TD_MAX_STEPS), ("rand", TD_MAX_STEPS), ("trained", CAP)])
def test_round_delta_is_the_per_game_replays_bit_for_bit(eng, orc, golden, net, cap):
    eng.set_weights(*golden_weights(golden("model.npz"), net))
    n = population_size(eng)
    pop = Population(eng, n, cap)
    delta = new_delta()
    st = eng.td_replay(LR, LAM, delta)
    grid = check_round(eng, orc, pop, delta, st, lambda s: (LR, LAM))
    assert n % grid and n // grid >= 6
    if cap < TD_MAX_STEPS:                                              # the cap truncates games, and some end right at it
        assert (pop.status == TRUNCATED).sum() > 0 and (pop.ply[pop.status == TRUNCATED] == cap).all()
        assert (pop.won & (pop.ply == cap)).sum() > 0
    else:
        assert pop.won.all()


@pytest.mark.gpu
@pytest.mark.parametrize("boundary", [30000, 40000])
def test_scheduled_round_is_the_per_game_replays_bit_for_bit(eng, orc, golden, boundary):
    """train.py:538 calls update_learning_params(games_done + k + 1) before the k-th game of a round (model.py:69-73).  The
    engine tabulates the schedule with the C library's pow, which is also what Python's float ** calls, so the per-game
    (lr, lambda) of the host and of the kernel are the same doubles and the round is exact across a schedule step."""
    from bgx.model import TDLGammonModel
    m = TDLGammonModel()

    def params(s):
        m.update_learning_params(games_done + s + 1)
        return m.learning_rate, m.lambda_decay
    eng.set_weights(*golden_weights(golden("model.npz"), "trained"))
    n = population_size(eng)
    pop = Population(eng, n, TD_MAX_STEPS)
    games_done = boundary - n // 2                                      # the round straddles the boundary
    assert len({params(s) for s in range(n)}) == 2
    delta = new_delta()
    st = eng.td_replay_scheduled(games_done, delta)
    check_round(eng, orc, pop, delta, st, params)


@pytest.mark.gpu
def test_second_round_replays_from_the_rebuilt_snapshot(eng, orc, golden):
    """apply_delta, then a new round from the new weights: its replay starts every game from the rebuilt snapshot."""
    w0 = golden_weights(golden("model.npz"), "trained")
    eng.set_weights(*w0)
    n = population_size(eng)
    pop = Population(eng, n, TD_MAX_STEPS)
    delta = new_delta()
    check_round(eng, orc, pop, delta, eng.td_replay(LR, LAM, delta), lambda s: (LR, LAM))
    eng.apply_delta(delta, 1.0 / n)
    assert not same_bits(eng.get_weights()[0], w0[0])
    eng.selfplay_next_round()
    eng.selfplay_round()
    pop.read(eng)
    delta2 = new_delta()
    check_round(eng, orc, pop, delta2, eng.td_replay(LR, LAM, delta2), lambda s: (LR, LAM))


@pytest.mark.gpu
def test_round_without_finished_games_is_zero(eng, golden):
    """In step mode finished games restart in place: no slot is ever won, so the replay has nothing to add."""
    eng.set_weights(*golden_weights(golden("model.npz"), "trained"))
    pop = Population(eng, population_size(eng), 64, play=False)
    eng.selfplay_step(40)
    rec, _, _ = eng.selfplay_read()
    assert not np.isin(rec[:, 31], (P1_WON, P2_WON, TRUNCATED)).any()
    delta = new_delta()
    st = eng.td_replay(LR, LAM, delta)
    got = delta.cpu().numpy()
    assert same_bits(got, np.zeros(NPARAMS_PADDED, np.float32))
    for k in ("td_steps", "games_finished", "truncated", "td_live_rows", "td_lazy_row_steps", "td_sq_error"):
        assert st[k] == 0, (k, st[k])
    assert len(rec) == pop.n


# ------------------------------------------------------------------ B. single games at the edges

PREFIXES = tuple(range(1, 19)) + (31, 32, 33, 257)
SETTINGS = [(lam, lr, won) for lam in (0.0, 0.5, 0.9, 1.0) for lr in (0.1, 1.0) for won in (True, False)]
# The 2,048-step game at lr 0.1 only: at lr 1 over 2,048 steps any two fp32 replays drift apart (measured on the B200: W1 rows
# of the kernel 100 ulps further from float64 than torch's), which says nothing about the kernel.
LONG_SETTINGS = [(lam, 0.1, k % 2 == 0) for k, lam in enumerate((0.0, 0.5, 0.9, 1.0))]

# Self-calibrated bounds against the float64 replay, measured on one B200 (1,000 W power limit) over every trajectory and setting
# of this section and the 256 fixture games:
#   per tensor, max|kernel - float64| <= TENSOR_A x max|torch - float64| + TENSOR_B ulp(max|w| of the tensor).  Kernel / torch:
#   median 1.00, p99 1.2 (W1, w2) and 1.7 (b1), max 1.3 - 2.1; with TENSOR_A = 2 the largest floor needed was 4.5 ulp (b2, one
#   number: T = 18, lambda 0.9, lr 1), every other tensor <= 0.1 ulp;
TENSOR_A, TENSOR_B = 2.0, 8.0
#   per W1 row f, max over units of |kernel - float64| <= ROW_A x torch's + ROW_B ulp(max|w0[:, f]|).  Kernel / torch over the
#   14,031 rows where torch is > 4 ulp off: median 1.00, p99 1.39, max 2.67; kernel up to 54 ulp off (p99 14); with ROW_A = 2
#   the largest floor needed was 3.3 ulp (fixture game 824, random-init).
ROW_A, ROW_B = 2.0, 8.0
SQ_TOL = 1e-5                            # per-step |delta| against torch, as test_gpu_parity holds it (measured: <= 4.8e-7)


@pytest.fixture(scope="module")
def games(eng, golden):
    """Real games: a greedy one of the trained net (>= 40 plies), and the first 2,048 records of a game under the `bar` tie
    net, which runs for thousands of plies (exported from a slot the 2,048-record cap truncated)."""
    eng.set_weights(*golden_weights(golden("model.npz"), "trained"))
    pop = Population(eng, 64, TD_MAX_STEPS)
    short = pop.trajs[int(np.flatnonzero(pop.won & (pop.ply >= 40))[0])]
    eng.set_weights(*tie_net("bar"))
    pop = Population(eng, 64, TD_MAX_STEPS)
    cut = np.flatnonzero(pop.status == TRUNCATED)
    assert len(cut) > 0
    long, _ = eng.export_trajectory(int(cut[0]))
    assert len(long) == TD_MAX_STEPS
    return short, long


def trajectory(games, T):
    short, long = games
    return short[:T] if T <= len(short) else long[:T]


def replay_three(eng, orc, w0, rec, won, lr, lam):
    """-> kernel, torch and float64 replays of one trajectory from w0: (flat new weights, squared TD errors) x 2, float64 flat"""
    from oracle.oracle import td_replay_f64
    from ref_td import replay_worker
    X = encode(orc, rec)
    eng.set_weights(*w0)
    new, sq = eng.td_replay_host(rec, won, lr, lam)
    t_new, t_sq = replay_worker((w0, X, int(won), lr, lam))
    w64 = np.concatenate([np.asarray(a, np.float64).reshape(-1) for a in td_replay_f64(w0, X, won, lr, lam)])
    return X, (flat(new), sq), (t_new, t_sq), w64


def edge_errors(w0, X, k_new, t_new, w64):
    """-> per tensor (kernel, torch, ulp) distances from float64; per W1 row (kernel, torch, ulp); rows whose feature is
    zero in every state"""
    w0 = flat(w0)
    ek, et = np.abs(k_new - w64), np.abs(t_new - w64)
    tensors = []
    for k in range(4):
        sl = slice(BOUNDS[k], BOUNDS[k + 1])
        scale = max(float(np.abs(w0[sl]).max()), float(np.abs(w64[sl]).max()))
        tensors.append((float(ek[sl].max()), float(et[sl].max()), float(np.spacing(np.float32(scale)))))
    rk, rt = ek[:BOUNDS[1]].reshape(128, 198).max(0), et[:BOUNDS[1]].reshape(128, 198).max(0)
    rulp = np.spacing(np.abs(w0[:BOUNDS[1]].reshape(128, 198)).max(0).astype(np.float32)).astype(np.float64)
    zero_rows = np.flatnonzero(~(X != 0).any(0))
    return tensors, (rk, rt, rulp), zero_rows


def check_edges(w0, X, kern, torch_, w64, what, per_tensor=True):
    (k_new, k_sq), (t_new, t_sq) = kern, torch_
    tensors, (rk, rt, rulp), zero_rows = edge_errors(w0, X, k_new, t_new, w64)
    for name, (ek, et, ulp) in zip(TENSORS, tensors):
        assert not per_tensor or ek <= TENSOR_A * et + TENSOR_B * ulp, (what, name, ek, et, ulp)
    bad = np.flatnonzero(rk > ROW_A * rt + ROW_B * rulp)
    assert len(bad) == 0, (what, "rows", bad[:8].tolist(), rk[bad[:4]].tolist(), rt[bad[:4]].tolist())
    # a row whose feature is zero in every state has no gradient: it comes back bit for bit
    W0 = flat(w0)[:BOUNDS[1]].reshape(128, 198)
    for new in (k_new, t_new):
        assert same_bits(new[:BOUNDS[1]].reshape(128, 198)[:, zero_rows], W0[:, zero_rows]), what
    assert len(k_sq) == len(t_sq) == len(X) - 1
    if len(k_sq):
        assert np.max(np.abs(np.sqrt(k_sq) - np.sqrt(t_sq))) <= SQ_TOL, (what, "TD errors")


@pytest.mark.gpu
@pytest.mark.parametrize("T", PREFIXES + (TD_MAX_STEPS,))
def test_single_game_edges_against_torch_and_float64(eng, orc, golden, games, T):
    """Prefixes of real games around the ring start (T = 1, 2, 3: the T > 1 / T > 2 guards and next_game's min(k, T - 1)), the
    record ring and the 4-step trips of td_replay_row (T = 4 .. 18, 31 .. 33), a long game (257) and the full c_k history
    (2,048), at lambda 0 and 1 (where the trips' padding lambda' = 1, c' = 0 meets a real step), lr 0.1 and 1, both outcomes."""
    w0 = golden_weights(golden("model.npz"), "trained")
    rec = trajectory(games, T)
    assert len(rec) == T
    for lam, lr, won in (SETTINGS if T < TD_MAX_STEPS else LONG_SETTINGS):
        X, kern, torch_, w64 = replay_three(eng, orc, w0, rec, won, lr, lam)
        check_edges(w0, X, kern, torch_, w64, (T, lam, lr, won))


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["rand", "trained"])
def test_per_row_errors_on_fixture_games(eng, orc, golden, tag):
    """Every W1 row of 128 fixture games per weight set (lr 0.1, lambda 0.9): a row that is live for a few steps only has a
    change far below its tensor's max|dw|, so a per-tensor metric would not see an error in it.  (The per-tensor distances of
    these games are test_gpu_parity's; one game's b1 / w2 / b2 can sit 100 ulp from float64 where torch is lucky.)"""
    from td_fixture import TdFixture
    fx = TdFixture(golden, tag)
    for g in range(0, fx.n, 8):
        rec = fx.trajectory(g)
        X, kern, torch_, w64 = replay_three(eng, orc, fx.w0, rec, bool(fx.p1_won[g]), fx.lr, fx.lam)
        check_edges(fx.w0, X, kern, torch_, w64, (tag, g), per_tensor=False)


@pytest.mark.gpu
def test_lr_zero_leaves_every_weight_bit_for_bit(eng, golden, games):
    for net in ("trained", "rand"):
        w0 = golden_weights(golden("model.npz"), net)
        eng.set_weights(*w0)
        for T in (1, 2, 3, 5, 17, 257, TD_MAX_STEPS):
            for lam in (0.0, 0.9, 1.0):
                new, _ = eng.td_replay_host(trajectory(games, T), T % 2 == 0, 0.0, lam)
                assert same_bits(flat(new), flat(w0)), (net, T, lam)


@pytest.mark.gpu
def test_trajectories_beyond_the_c_k_history_are_refused(eng, golden, games):
    from bgx import lib as L
    eng.set_weights(*golden_weights(golden("model.npz"), "trained"))
    long = games[1]
    with pytest.raises(L.BgxError) as e:
        eng.td_replay_host(np.concatenate([long, long[-1:]]), True, LR, LAM)
    assert e.value.code == L.E_INVALID
    Population(eng, 8, TD_MAX_STEPS + 1, play=False)
    for call in (lambda d: eng.td_replay(LR, LAM, d), lambda d: eng.td_replay_scheduled(0, d)):
        with pytest.raises(L.BgxError) as e:
            call(new_delta())
        assert e.value.code == L.E_INVALID


# ------------------------------------------------------------------ C. the kernel's feature values over their whole domain

def feature_domains():
    """Every value each of the 198 features can take (model.py:111-144, float32)"""
    step = {0.0, 1.0}
    ramp = {0.0} | {float(np.float32((c - 3) / 2.0)) for c in range(4, 16)}
    dom = []
    for f in range(192):
        dom.append(ramp if f % 4 == 3 else step)
    dom += [step, step]
    dom += [{float(np.float32(b / 2.0)) for b in range(16)}] * 2
    dom += [{float(np.float32(k / 15.0)) for k in range(16)}] * 2
    return dom


def synthetic_records():
    """Valid boards (15 checkers a side between points, bar and borne off; no point held by both) that between them take
    every point byte -15 .. 15 on every point, every bar and borne-off count 0 .. 15 of either side and both turn flags,
    plus mixed random boards; shuffled into one trajectory, the turn flag alternating."""
    rng = np.random.default_rng(2026)
    boards = []
    for v in range(1, 16):                                   # v checkers of PLAYER1 on point i, v of PLAYER2 on point i + 12
        for i in range(24):
            b = np.zeros(28, np.int64)
            b[i], b[(i + 12) % 24] = v, -v
            rest = 15 - v
            b[24], b[26] = rest // 2, rest - rest // 2
            b[25], b[27] = rest - rest // 2, rest // 2
            boards.append(b)
    for k in range(16):                                      # bar k / borne off 15 - k, and the mirror for PLAYER2
        b = np.zeros(28, np.int64)
        b[24], b[26], b[25], b[27] = k, 15 - k, 15 - k, k
        boards.append(b)
    for _ in range(64):                                      # mixed boards: each side spread over its own points, bar, off
        b = np.zeros(28, np.int64)
        pts = rng.permutation(24)
        for side, mine in ((1, pts[:12]), (-1, pts[12:])):
            where = rng.choice(np.concatenate([mine, [24 if side > 0 else 25, 26 if side > 0 else 27]]), 15)
            for p in where:
                b[p] += side if p < 24 else 1
        boards.append(b)
    boards = np.array(boards)[rng.permutation(len(boards))]
    rec = np.zeros((len(boards), 32), np.int8)
    rec[:, :28] = boards
    rec[:, 28] = np.arange(len(boards)) % 2
    return rec


def test_synthetic_boards_cover_every_feature_value(orc):
    rec = synthetic_records()
    st = rec[:, :28].astype(np.int64)
    p1 = np.where(st[:, :24] > 0, st[:, :24], 0).sum(1) + st[:, 24] + st[:, 26]
    p2 = np.where(st[:, :24] < 0, -st[:, :24], 0).sum(1) + st[:, 25] + st[:, 27]
    assert (p1 == 15).all() and (p2 == 15).all() and (st[:, 24:28] >= 0).all()
    for i in range(24):
        assert set(st[:, i].tolist()) == set(range(-15, 16)), i
    for i in range(24, 28):
        assert set(st[:, i].tolist()) == set(range(16)), i
    assert set(rec[:, 28].tolist()) == {0, 1}
    X = encode(orc, rec)
    for f, dom in enumerate(feature_domains()):
        assert set(X[:, f].astype(np.float64).tolist()) == dom, f


# |sqrt(sq[t]) - |V64(s_t+1) - V64(s_t)|| over the 440 synthetic states, measured on one B200 (1,000 W): max 9.7e-8 random-init,
# 1.2e-7 trained (median 2.6e-8 / 2.8e-8); the smallest |V(s_t+1) - V(s_t)| among the pairs is 8.2e-7 / 1.4e-3
VALUE_TOL = 5e-7


@pytest.mark.gpu
@pytest.mark.parametrize("net", ["rand", "trained"])
def test_kernel_feature_values_over_their_whole_domain(eng, orc, golden, net):
    """At lr = 0 the weights never change, so the replay's squared TD error of step t is (V(s_t+1) - V(s_t))^2 under the
    snapshot, with the values the kernel computed from its own features: compared with float64 on every consecutive pair.
    A wrong feature value moves V by ~1e-3."""
    w0 = golden_weights(golden("model.npz"), net)
    rec = synthetic_records()
    eng.set_weights(*w0)
    new, sq = eng.td_replay_host(rec, True, 0.0, LAM)
    assert same_bits(flat(new), flat(w0))
    v = forward64(w0, encode(orc, rec))
    err = np.abs(np.sqrt(sq) - np.abs(np.diff(v)))
    assert err.max() <= VALUE_TOL, (net, float(err.max()), int(np.argmax(err)))
