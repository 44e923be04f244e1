"""Batched head-to-head play on one GPU: the reference's evaluation loops
(`_play_head_to_head` / `evaluate_parallel`, train.py:262-302; `play_vs_random` / `play_vs_model`,
benchmark.py:64-130) for thousands of games at once.

All games advance in lockstep, one ply per iteration: the games whose mover is played by policy A
go through one `bgx_select_moves` launch of engine A, the others through engine B, then `bgx_advance`
checks for the end of the game, flips the mover and rolls the next dice (Philox, the self-play dice
rule, so every game can be replayed into the reference through `Game.setDice`).  A policy is a
weight tuple (greedy, epsilon = 0: `make_move`), the string "random" (`_random_move`,
benchmark.py:54-61: a uniformly random legal sequence) or a `TwoPly` (the same net looking one roll
ahead: `bgx_select_moves_2ply`).
"""
import numpy as np
import torch

from .engine import BatchEngine
from .synth import START_BOARD

RANDOM = "random"


class TwoPly:
    """Two-ply policy: `weights` looking one roll ahead (BatchEngine.select_moves_2ply); `candidates` = how many of the best
    one-ply afterstates are expanded (0 = all of them)."""

    def __init__(self, weights, candidates=0):
        if int(candidates) < 0:
            raise ValueError("candidates must be >= 0")
        self.weights = weights
        self.candidates = int(candidates)


class Arena:
    """Two engines on one device, one per policy, sharing the device buffers of the match."""

    def __init__(self, device=0):
        self.device = torch.device("cuda", device)
        self.eng = [BatchEngine(device), BatchEngine(device)]
        stream = torch.cuda.current_stream(self.device).cuda_stream
        for e in self.eng:
            e.set_stream(stream)
        self._dummy = None

    def close(self):
        for e in self.eng:
            e.close()

    def _load(self, k, policy):
        """-> (epsilon, two-ply candidates or None) of the policy now loaded into engine k"""
        if isinstance(policy, TwoPly):
            self.eng[k].set_weights(*policy.weights)
            return 0.0, policy.candidates
        if isinstance(policy, str):
            if policy != RANDOM:
                raise ValueError(policy)
            if self._dummy is None:
                self._dummy = (np.zeros((128, 198), np.float32), np.zeros(128, np.float32),
                               np.zeros((1, 128), np.float32), np.zeros(1, np.float32))
            self.eng[k].set_weights(*self._dummy)       # the random policy never evaluates
            return 1.0, None
        self.eng[k].set_weights(*policy)
        return 0.0, None

    def play(self, policy_a, policy_b, side_of_a, first_mover, seed=0x5EED2026, max_plies=4096, record=False):
        """n games; game i: policy A plays PLAYER `side_of_a[i]` (0/1), PLAYER `first_mover[i]` moves first.
        -> dict(winner int8[n] (0/1, -1 if max_plies ran out), plies int32[n], log=[(ply, idx, query, chosen)] if record)"""
        dev = self.device
        side = torch.as_tensor(np.asarray(side_of_a), dtype=torch.int8, device=dev)
        n = side.numel()
        (eps_a, two_a), (eps_b, two_b) = self._load(0, policy_a), self._load(1, policy_b)
        eps, two = [eps_a, eps_b], [two_a, two_b]
        start = np.zeros((n, 32), np.int8)
        start[:, :24] = START_BOARD
        start[:, 28] = np.asarray(first_mover, np.int8) ^ 1           # bgx_advance flips it and rolls ply 0
        rec = torch.from_numpy(start).to(dev)
        gid = torch.arange(n, dtype=torch.int64, device=dev)
        self.eng[0].advance(rec, rec, seed, 0, gid, None)
        winner = torch.full((n,), -1, dtype=torch.int8, device=dev)
        plies = torch.zeros(n, dtype=torch.int32, device=dev)
        alive = gid.clone()
        log = []
        for ply in range(max_plies):
            if alive.numel() == 0:
                break
            a_moves = rec[alive, 28] == side[alive]
            for k, mask in ((0, a_moves), (1, ~a_moves)):
                idx = alive[mask]
                m = idx.numel()
                if m == 0:
                    continue
                q = rec[idx].contiguous()
                ch = torch.empty_like(q)
                if two[k] is not None:
                    self.eng[k].select_moves_2ply(q, two[k], chosen=ch)
                else:
                    self.eng[k].select_moves(q, epsilon=eps[k], seed=(seed ^ ((ply + 1) << 32)) & (2 ** 64 - 1), chosen=ch)
                w = torch.empty(m, dtype=torch.int8, device=dev)
                nxt = torch.empty_like(q)
                self.eng[k].advance(ch, nxt, seed, ply + 1, idx, w)
                rec[idx] = nxt
                winner[idx] = w
                plies[idx] += 1
                if record:
                    log.append((ply, idx.cpu().numpy(), q.cpu().numpy(), ch.cpu().numpy()))
            alive = alive[winner[alive] < 0]
        out = {"winner": winner.cpu().numpy(), "plies": plies.cpu().numpy()}
        if record:
            out["log"] = log
        return out


def evaluate(arena, cur_weights, opp_weights, num_games=100, seed=0x5EED2026):
    """evaluate_parallel (train.py:295-301): win rate of the current model against an opponent, sides
    alternated (A is PLAYER1 in even games); `Game(game_idx % 2)` seats the first mover (train.py:265)."""
    i = np.arange(num_games)
    side = (i % 2).astype(np.int8)                   # a_is_p1 = (i % 2 == 0)
    res = arena.play(cur_weights, opp_weights, side, i % 2, seed=seed)
    return float(np.mean(res["winner"] == side))


def play_vs_random(arena, weights, num_games, seed=0x5EED2026):
    """benchmark.py:64-96: the model as PLAYER1 against the random policy, alternating who starts.
    -> (model win rate, average game length in plies as the reference counts them)"""
    i = np.arange(num_games)
    res = arena.play(weights, RANDOM, np.zeros(num_games, np.int8), i % 2, seed=seed)
    return float(np.mean(res["winner"] == 0)), float(np.mean(res["plies"] - 1))


def play_vs_model(arena, weights1, weights2, num_games, seed=0x5EED2026):
    """benchmark.py:99-130: model1 as PLAYER1 against model2, alternating who starts."""
    i = np.arange(num_games)
    res = arena.play(weights1, weights2, np.zeros(num_games, np.int8), i % 2, seed=seed)
    return float(np.mean(res["winner"] == 0)), float(np.mean(res["plies"] - 1))
