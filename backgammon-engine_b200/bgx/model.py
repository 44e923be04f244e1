"""TDLGammonModel — the reference's model contract (pysrc/TD(λ) model/model.py:31-222) with the
batched GPU engine behind it.

Kept from the reference, so train.py / benchmark.py / play_model.py / tests.py keep working
when they import this class instead: constructor without arguments, `fc1`/`fc2` parameter
names and shapes (state_dict compatible with models/*.pth), `learning_rate`, `lambda_decay`,
`eligibility_traces`, and the methods `forward`, `update_learning_params`, `encode_state`,
`encode_state_np`, `_encode_states_np`, `select_best_action`, `_simulate_sequence`,
`make_move`, `initialize_traces`, `initialize_weights`.

Added: `engine()` (a BatchEngine holding these weights), `make_moves_batch` (batched
make_move over many games at once, greedy or two-ply), `rollout_batch` (rollout values of many
positions) — the per-object `make_move` stays a host-side loop because
one position per call cannot amortise a kernel launch; the batch calls are the fast path.
"""
import random

import numpy as np
import torch
import torch.nn as nn

import backgammon_env as bg  # the libbgx-backed compat module (backgammon-engine_b200/lib)

P1 = int(bg.PlayerType.PLAYER1)


def encode_rows(states, turn):
    """float32[N,198] encoding of int[N,28] rows (model.py:111-144), vectorised over points."""
    states = np.asarray(states)
    n_rows = states.shape[0]
    board = states[:, :24].astype(np.int64)
    count = np.abs(board)
    X = np.zeros((n_rows, 24, 8), dtype=np.float32)
    unit = np.stack([count >= 1, count >= 2, count >= 3], axis=2).astype(np.float32)
    extra = np.where(count >= 4, (count - 3) / 2, 0.0).astype(np.float32)
    feats = np.concatenate([unit, extra[:, :, None]], axis=2)            # [N,24,4]
    mine = (board > 0)[:, :, None]
    X[:, :, 0:4] = np.where(mine, feats, 0.0)
    X[:, :, 4:8] = np.where(mine, 0.0, feats)
    out = np.zeros((n_rows, 198), dtype=np.float32)
    out[:, :192] = X.reshape(n_rows, 192)
    p1_turn = turn == bg.PlayerType.PLAYER1
    out[:, 192] = 1.0 if p1_turn else 0.0
    out[:, 193] = 0.0 if p1_turn else 1.0
    out[:, 194] = states[:, 24] / 2
    out[:, 195] = states[:, 25] / 2
    out[:, 196] = states[:, 26] / 15.0
    out[:, 197] = states[:, 27] / 15.0
    return out


class TDLGammonModel(nn.Module):
    def __init__(self, input_size=198, hidden_size=128):
        super().__init__()
        self.fc1 = nn.Linear(input_size, hidden_size)
        self.fc2 = nn.Linear(hidden_size, 1)
        self.learning_rate = 0.1
        self.initialize_weights()
        self.eligibility_traces = {}
        self.initialize_traces()
        self.lambda_decay = 0.7
        self._engine = None
        self._uploaded = None
        self._ahead = None                                   # a GpuTrainer whose weights are newer than this module's

    # ------------------------------------------------------------------ reference contract
    def initialize_traces(self):
        self.eligibility_traces = {name: torch.zeros_like(p.data) for name, p in self.named_parameters() if p.requires_grad}

    def initialize_weights(self):
        for m in self.modules():
            if isinstance(m, nn.Linear):
                nn.init.xavier_uniform_(m.weight, gain=0.1)
                if m.bias is not None:
                    nn.init.constant_(m.bias, 0)

    def forward(self, x):
        return torch.sigmoid(self.fc2(torch.sigmoid(self.fc1(x))))

    def update_learning_params(self, episode):
        self.learning_rate = max(0.01, 0.1 * (0.96 ** (episode // 40000)))
        self.lambda_decay = max(0.7, 0.9 * (0.96 ** (episode // 30000)))

    def _encode_states_np(self, states, turn):
        return encode_rows(states, turn)

    def encode_state_np(self, game):
        row = np.empty((1, 28), dtype=np.int64)
        row[0, :24] = game.getGameBoard()
        row[0, 24] = game.getJailedCount(bg.PlayerType.PLAYER1)
        row[0, 25] = game.getJailedCount(bg.PlayerType.PLAYER2)
        row[0, 26] = game.getBornOffCount(bg.PlayerType.PLAYER1)
        row[0, 27] = game.getBornOffCount(bg.PlayerType.PLAYER2)
        return encode_rows(row, game.getTurn())[0]

    def encode_state(self, game):
        return torch.from_numpy(self.encode_state_np(game))

    def _simulate_sequence(self, sim_game, seq):
        for o, dst in seq:
            player = sim_game.getPlayers(sim_game.getTurn())
            ok, _ = sim_game.tryMove(player, int(abs(o - dst)), o, dst)
            if not ok:
                return False
        return True

    def select_best_action(self, game, actions):
        device = next(self.parameters()).device
        p1 = game.getTurn() == bg.PlayerType.PLAYER1
        values = []
        for seq in actions:
            sim = game.clone()
            if not self._simulate_sequence(sim, seq):
                values.append(float("-inf") if p1 else float("inf"))
                continue
            with torch.no_grad():
                values.append(self(self.encode_state(sim).to(device).unsqueeze(0)).item())
        pick = max if p1 else min
        return actions[pick(range(len(values)), key=values.__getitem__)]

    def make_move(self, game, game_idx: int = 1, epsilon: float = 0.0):
        """One ply on a compat Game object: same decisions as model.py:180-222."""
        self.eval()
        turn = game.getTurn()
        mover = game.getPlayers(turn)
        d = game.get_last_dice()
        actions, states = game.evaluateTurnSequences(turn, d[0], d[1])
        if not actions:
            return []
        if epsilon > 0.0 and random.random() < epsilon:
            idx = random.randrange(len(actions))
        else:
            device = next(self.parameters()).device
            X = torch.from_numpy(encode_rows(states, turn)).to(device)
            with torch.inference_mode():
                values = self(X).squeeze(1)
            idx = int(torch.argmax(values) if turn == bg.PlayerType.PLAYER1 else torch.argmin(values))
        best = actions[idx]
        for o, dst in best:
            game.tryMove(mover, int(abs(o - dst)), o, dst)
        return best

    # ------------------------------------------------------------------ GPU fast paths
    def weights_np(self):
        sd = self.state_dict()
        return tuple(sd[k].detach().cpu().numpy() for k in ("fc1.weight", "fc1.bias", "fc2.weight", "fc2.bias"))

    def _weights_version(self):
        """Changes whenever a parameter is written (in place or replaced): what tells engine() to upload again."""
        return tuple((p.data_ptr(), p._version) for p in (self.fc1.weight, self.fc1.bias, self.fc2.weight, self.fc2.bias))

    def engine(self, device=0):
        """BatchEngine on `device` holding this module's weights (created on first use; raises without a GPU).  The weights
        are uploaded when the engine is created and again only after the module's parameters have changed."""
        from .engine import BatchEngine
        if self._engine is None:
            self._engine = BatchEngine(device)
            self._uploaded = None
        version = self._weights_version()
        if version != self._uploaded:
            self._engine.set_weights(*self.weights_np())
            self._uploaded = version
        return self._engine

    def load_weights_from(self, engine):
        """Copy an engine's weights (e.g. a GpuTrainer's after its rounds) into this module."""
        W1, b1, w2, b2 = engine.get_weights()
        with torch.no_grad():
            self.fc1.weight.copy_(torch.from_numpy(W1)); self.fc1.bias.copy_(torch.from_numpy(b1))
            self.fc2.weight.copy_(torch.from_numpy(w2)); self.fc2.bias.copy_(torch.from_numpy(b2))

    def load_engine_weights(self):
        """Copy this module's own engine weights back into the module."""
        self.load_weights_from(self._engine)
        self._uploaded = self._weights_version()

    def make_moves_batch(self, games, epsilon=0.0, seed=0, device=0, plies=1, candidates=0):
        """make_move for a list of compat Game objects in ONE kernel launch; applies the chosen
        sequences to the games and returns them (list[list[tuple]]).  plies=2 looks one roll ahead
        (BatchEngine.select_moves_2ply_host; `candidates` = how many of the best one-ply afterstates
        are expanded, 0 = all); it has no exploration, so epsilon must be 0 there."""
        if plies not in (1, 2):
            raise ValueError(f"plies must be 1 or 2, not {plies}")
        if plies == 2 and epsilon > 0.0:
            raise ValueError("two-ply move selection has no epsilon exploration")
        q = _game_records(games)
        if plies == 2:
            out = self.engine(device).select_moves_2ply_host(q, max_candidates=candidates)
        else:
            out = self.engine(device).select_moves_host(q, epsilon=epsilon, seed=seed)
        result = []
        for i, g in enumerate(games):
            seq = [(int(o), int(d)) for o, d in out["moves"][i, : out["moves_len"][i]]]
            mover = g.getPlayers(g.getTurn())
            for o, d in seq:
                g.tryMove(mover, abs(o - d), o, d)
            result.append(seq)
        return result

    def rollout_batch(self, games, trials=1296, max_plies=0, seed=0x5EED2026, device=0, vr_plies=0):
        """Rollouts of compat Game objects (BatchEngine.rollout_host, DESIGN 7d): `trials` greedy games from each game's
        position with its player on roll (the dice are ignored), stratified over the first roll when trials is a multiple of 36,
        cut after `max_plies` plies (0: played to the end).  The games are not modified.
        -> dict(p1_win f64[n] = P(PLAYER1 wins), std_err f64[n], outcomes f64[n, 6] = fractions of PLAYER1 single / gammon /
        backgammon and PLAYER2 single / gammon / backgammon wins).  vr_plies > 0 (DESIGN 7e) adds vr_p1_win and vr_std_err, the
        luck-adjusted estimate over the first vr_plies plies of each trial and its standard error."""
        trials = int(trials)
        out = self.engine(device).rollout_host(_game_records(games), trials, max_plies=max_plies, seed=seed,
                                               stratify=trials % 36 == 0, vr_plies=vr_plies)
        r = {"p1_win": out["mean"], "std_err": out["std_err"], "outcomes": out["counts"][:, :6] / float(trials)}
        if vr_plies:
            r["vr_p1_win"], r["vr_std_err"] = out["vr_mean"], out["vr_std_err"]
        return r


def _game_records(games):
    """RECORDs of compat Game objects: position, player on roll, the dice last rolled"""
    q = np.zeros((len(games), 32), np.int8)
    for i, g in enumerate(games):
        q[i, :24] = g.getGameBoard()
        q[i, 24], q[i, 25] = g.getJailedCount(0), g.getJailedCount(1)
        q[i, 26], q[i, 27] = g.getBornOffCount(0), g.getBornOffCount(1)
        q[i, 28] = g.getTurn()
        q[i, 29:31] = g.get_last_dice()
    return q
