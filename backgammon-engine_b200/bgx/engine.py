"""BatchEngine — the batched GPU entry points of libbgx behind one Python object.

Two flavours of every call, mirroring the C-ABI:
  * `*_host`  numpy in / numpy out; the library does the H2D/D2H copies (the end-to-end path)
  * device    torch CUDA tensors in / out (raw pointers are handed to the library, which only
              enqueues kernels on the engine's stream)
PyTorch is plumbing here (device memory, streams, torch.distributed); all compute is the
library's hand-written sm_100a kernels.
"""
import ctypes as C

import numpy as np

from . import lib as L


def _records(a):
    a = np.ascontiguousarray(a, dtype=np.int8)
    if a.ndim != 2 or a.shape[1] != 32:
        raise ValueError("records are int8[n, 32]")
    return a


class BatchEngine:
    def __init__(self, device=0):
        self._lib = L.load()
        h = C.c_void_p()
        L.check(self._lib.bgx_create(int(device), C.byref(h)))
        self._h = h
        self.device = int(device)

    def close(self):
        if getattr(self, "_h", None):
            self._lib.bgx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ plumbing
    def set_stream(self, cuda_stream):
        """cuda_stream: integer cudaStream_t (e.g. torch.cuda.current_stream().cuda_stream)"""
        L.check(self._lib.bgx_set_stream(self._h, C.c_void_p(int(cuda_stream) or None)))

    def synchronize(self):
        L.check(self._lib.bgx_synchronize(self._h))

    def set_weights(self, W1, b1, w2, b2):
        """state_dict tensors (model.py:36-37): fc1.weight[128,198], fc1.bias[128], fc2.weight[1,128], fc2.bias[1]"""
        arrs = [np.ascontiguousarray(np.asarray(a, dtype=np.float32)).reshape(-1) for a in (W1, b1, w2, b2)]
        assert [a.size for a in arrs] == [128 * 198, 128, 128, 1], "weight shapes"
        L.check(self._lib.bgx_set_weights(self._h, *(a.ctypes.data for a in arrs)))

    def get_weights(self):
        W1 = np.zeros((128, 198), np.float32)
        b1 = np.zeros(128, np.float32)
        w2 = np.zeros((1, 128), np.float32)
        b2 = np.zeros(1, np.float32)
        L.check(self._lib.bgx_get_weights(self._h, W1.ctypes.data, b1.ctypes.data, w2.ctypes.data, b2.ctypes.data))
        return W1, b1, w2, b2

    def launch_count(self):
        n = C.c_int64()
        L.check(self._lib.bgx_launch_count(self._h, C.byref(n)))
        return n.value

    def last_kernel_ms(self):
        ms = C.c_float()
        L.check(self._lib.bgx_last_kernel_ms(self._h, C.byref(ms)))
        return ms.value

    def kernel_config(self):
        a, b = C.c_int(), C.c_int()
        L.check(self._lib.bgx_kernel_config(self._h, C.byref(a), C.byref(b)))
        return {"k_selfplay": a.value, "k_select": b.value}

    def sfu_monotone(self):
        """Violations of monotonicity of ex2.approx / rcp.approx on this device (bgx_sfu_monotone): both must be 0."""
        a, b = C.c_int64(), C.c_int64()
        L.check(self._lib.bgx_sfu_monotone(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def set_option(self, key, value):
        """Tuning knobs of the fused ply kernels (bgx_set_option): selfplay_warps, select_warps, select_lane_grid, ..."""
        L.check(self._lib.bgx_set_option(self._h, key.encode(), int(value)))

    def device_props(self):
        sm, khz, mem = C.c_int(), C.c_int(), C.c_int64()
        L.check(self._lib.bgx_device_props(self._h, C.byref(sm), C.byref(khz), C.byref(mem)))
        return {"sm_count": sm.value, "clock_khz": khz.value, "global_mem": mem.value}

    # ------------------------------------------------------------------ enumeration
    def enumerate_summary_host(self, queries):
        q = _records(queries)
        n = q.shape[0]
        n_seq, n_unique, digest = np.zeros(n, np.int32), np.zeros(n, np.int32), np.zeros(n, np.uint64)
        L.check(self._lib.bgx_enumerate_summary_host(self._h, q.ctypes.data, n, n_seq.ctypes.data,
                                                     n_unique.ctypes.data, digest.ctypes.data))
        return n_seq, n_unique, digest

    def enumerate_summary(self, queries, n_seq, n_unique, digest):
        """device tensors: int8[n,32] -> int32[n], int32[n], int64[n] (digest bits)"""
        L.check(self._lib.bgx_enumerate_summary(self._h, L.ptr(queries), queries.shape[0], L.ptr(n_seq),
                                                L.ptr(n_unique), L.ptr(digest)))

    def enumerate_host(self, queries, cap=None):
        """-> offsets int64[n+1], moves int8[R,4,2], lens int8[R], states int8[R,32]"""
        q = _records(queries)
        n = q.shape[0]
        offsets = np.zeros(n + 1, np.int64)
        total = C.c_int64()
        cap = int(cap) if cap else max(1024, 128 * n)
        while True:
            mv = np.zeros((cap, 4, 2), np.int8)
            ln = np.zeros(cap, np.int8)
            st = np.zeros((cap, 32), np.int8)
            rc = self._lib.bgx_enumerate_host(self._h, q.ctypes.data, n, cap, offsets.ctypes.data, mv.ctypes.data,
                                              ln.ctypes.data, st.ctypes.data, C.byref(total))
            if rc == L.E_CAPACITY:
                cap = int(total.value)
                continue
            L.check(rc)
            t = total.value
            return offsets, mv[:t], ln[:t], st[:t]

    def enumerate_count(self, queries, n_seq, offsets):
        """device tensors: int8[n,32] -> int32[n] list sizes, int64[n+1] exclusive prefix sum (offsets[n] = total rows)"""
        L.check(self._lib.bgx_enumerate_count(self._h, L.ptr(queries), queries.shape[0], L.ptr(n_seq), L.ptr(offsets)))

    def enumerate(self, queries, offsets, moves, lens, states):
        L.check(self._lib.bgx_enumerate(self._h, L.ptr(queries), queries.shape[0], L.ptr(offsets), L.ptr(moves),
                                        L.ptr(lens), L.ptr(states)))

    # ------------------------------------------------------------------ encode / evaluate
    def encode_host(self, records):
        r = _records(records)
        X = np.zeros((r.shape[0], 198), np.float32)
        L.check(self._lib.bgx_encode_host(self._h, r.ctypes.data, r.shape[0], X.ctypes.data))
        return X

    def encode(self, records, X):
        L.check(self._lib.bgx_encode(self._h, L.ptr(records), records.shape[0], L.ptr(X)))

    def evaluate_host(self, records):
        r = _records(records)
        V = np.zeros(r.shape[0], np.float32)
        L.check(self._lib.bgx_evaluate_host(self._h, r.ctypes.data, r.shape[0], V.ctypes.data))
        return V

    def evaluate(self, records, V):
        L.check(self._lib.bgx_evaluate(self._h, L.ptr(records), records.shape[0], L.ptr(V)))

    # ------------------------------------------------------------------ batched make_move
    def select_moves_host(self, queries, epsilon=0.0, seed=0, out=None):
        """-> dict(chosen int8[n,32], moves int8[n,4,2], moves_len int8[n], value f32[n], n_seq, n_scored)
        `out` may carry preallocated (e.g. pinned) numpy arrays under the same keys."""
        q = _records(queries)
        n = q.shape[0]
        o = out or {}
        o.setdefault("chosen", np.zeros((n, 32), np.int8))
        o.setdefault("moves", np.zeros((n, 4, 2), np.int8))
        o.setdefault("moves_len", np.zeros(n, np.int8))
        o.setdefault("value", np.zeros(n, np.float32))
        o.setdefault("n_seq", np.zeros(n, np.int32))
        o.setdefault("n_scored", np.zeros(n, np.int32))
        L.check(self._lib.bgx_select_moves_host(self._h, q.ctypes.data, n, float(epsilon), int(seed),
                                                L.ptr(o["chosen"]), L.ptr(o["moves"]), L.ptr(o["moves_len"]),
                                                L.ptr(o["value"]), L.ptr(o["n_seq"]), L.ptr(o["n_scored"])))
        return o

    def select_moves_host_async(self, lane, queries, out, epsilon=0.0, seed=0):
        """Queue one batch on `lane` (0..3) and return; `out` maps output names to preallocated
        (ideally pinned) numpy arrays, missing names are not computed.  wait(lane) completes it."""
        q = _records(queries)
        L.check(self._lib.bgx_select_moves_host_async(self._h, int(lane), q.ctypes.data, q.shape[0], float(epsilon), int(seed),
                                                      L.ptr(out.get("chosen")), L.ptr(out.get("moves")), L.ptr(out.get("moves_len")),
                                                      L.ptr(out.get("value")), L.ptr(out.get("n_seq")), L.ptr(out.get("n_scored"))))

    def play_ply_host_async(self, lane, records, next_ply, game_id, next_records, winner=None, value=None, n_seq=None,
                            epsilon=0.0, explore_seed=0, dice_seed=0x5EED2026):
        """One iteration of play_game's loop (train.py:103-121) for a batch of games through (pinned) numpy buffers:
        make_move + is_game_over + setTurn + roll_dice of ply next_ply[i] of game game_id[i].  wait(lane) completes it."""
        q = _records(records)
        n = q.shape[0]
        assert next_records.dtype == np.int8 and next_records.shape == (n, 32) and next_records.flags["C_CONTIGUOUS"]
        assert next_ply is None or (next_ply.dtype == np.int32 and next_ply.shape == (n,) and next_ply.flags["C_CONTIGUOUS"])
        assert game_id is None or (game_id.dtype == np.int64 and game_id.shape == (n,) and game_id.flags["C_CONTIGUOUS"])
        L.check(self._lib.bgx_play_ply_host_async(self._h, int(lane), q.ctypes.data, L.ptr(next_ply), L.ptr(game_id), n,
                                                  float(epsilon), int(explore_seed), int(dice_seed),
                                                  L.ptr(next_records), L.ptr(winner), L.ptr(value), L.ptr(n_seq)))

    def play_ply_restart_host_async(self, lane, records, ply, game_id, id_stride, next_records, winner=None, value=None, n_seq=None,
                                    first_mover=L.FIRST_PARITY, epsilon=0.0, explore_seed=0, dice_seed=0x5EED2026):
        """play_ply_host_async with the bookkeeping on the device: ply / game_id (int32 / int64 numpy, updated in place when the
        lane completes) describe `records` on entry and `next_records` on return; finished games restart in place."""
        q = _records(records)
        n = q.shape[0]
        assert next_records.dtype == np.int8 and next_records.shape == (n, 32) and next_records.flags["C_CONTIGUOUS"]
        assert ply.dtype == np.int32 and ply.shape == (n,) and ply.flags["C_CONTIGUOUS"]
        assert game_id.dtype == np.int64 and game_id.shape == (n,) and game_id.flags["C_CONTIGUOUS"]
        L.check(self._lib.bgx_play_ply_restart_host_async(self._h, int(lane), q.ctypes.data, L.ptr(ply), L.ptr(game_id), int(id_stride),
                                                          int(first_mover), n, float(epsilon), int(explore_seed), int(dice_seed),
                                                          L.ptr(next_records), L.ptr(winner), L.ptr(value), L.ptr(n_seq)))

    def wait(self, lane):
        L.check(self._lib.bgx_lane_wait(self._h, int(lane)))

    def advance(self, chosen, nxt, seed, ply, game_id=None, winner=None):
        """device tensors: afterstates int8[n,32] -> next queries (mover flipped, dice of `ply` rolled, byte 31 = result)"""
        L.check(self._lib.bgx_advance(self._h, L.ptr(chosen), L.ptr(nxt), chosen.shape[0], int(seed), int(ply),
                                      L.ptr(game_id), L.ptr(winner)))

    def select_moves(self, queries, epsilon=0.0, seed=0, chosen=None, moves=None, moves_len=None, value=None,
                     n_seq=None, n_scored=None):
        L.check(self._lib.bgx_select_moves(self._h, L.ptr(queries), queries.shape[0], float(epsilon), int(seed),
                                           L.ptr(chosen), L.ptr(moves), L.ptr(moves_len), L.ptr(value),
                                           L.ptr(n_seq), L.ptr(n_scored)))

    def select_moves_2ply_host(self, queries, max_candidates=0, out=None):
        """Two-ply move selection (bgx_select_moves_2ply): every distinct afterstate, or the `max_candidates` best by one-ply
        value, valued by the expectation over the opponent's 21 rolls of the opponent's greedy reply.
        -> dict(chosen int8[n,32], moves int8[n,4,2], moves_len int8[n], value f32[n], n_candidates int32[n], n_expanded int32[n])"""
        q = _records(queries)
        n = q.shape[0]
        o = out or {}
        o.setdefault("chosen", np.zeros((n, 32), np.int8))
        o.setdefault("moves", np.zeros((n, 4, 2), np.int8))
        o.setdefault("moves_len", np.zeros(n, np.int8))
        o.setdefault("value", np.zeros(n, np.float32))
        o.setdefault("n_candidates", np.zeros(n, np.int32))
        o.setdefault("n_expanded", np.zeros(n, np.int32))
        L.check(self._lib.bgx_select_moves_2ply_host(self._h, q.ctypes.data, n, int(max_candidates),
                                                     L.ptr(o["chosen"]), L.ptr(o["moves"]), L.ptr(o["moves_len"]),
                                                     L.ptr(o["value"]), L.ptr(o["n_candidates"]), L.ptr(o["n_expanded"])))
        return o

    def select_moves_2ply(self, queries, max_candidates=0, chosen=None, moves=None, moves_len=None, value=None,
                          n_candidates=None, n_expanded=None):
        """select_moves_2ply_host on device tensors (the engine's stream)"""
        L.check(self._lib.bgx_select_moves_2ply(self._h, L.ptr(queries), queries.shape[0], int(max_candidates),
                                                L.ptr(chosen), L.ptr(moves), L.ptr(moves_len), L.ptr(value),
                                                L.ptr(n_candidates), L.ptr(n_expanded)))

    def rollout_host(self, positions, trials, max_plies=0, seed=0x5EED2026, stratify=True, per_trial=False):
        """Rollouts (bgx_rollout, DESIGN 7d): `trials` greedy games from every position (int8[n, 32], byte 28 = player on roll),
        cut after `max_plies` plies (0: played to the end).
        -> dict(mean f64[n], std_err f64[n], counts int64[n, 8]) and, with per_trial, trial_value f32[n, trials],
        trial_outcome int8[n, trials], trial_plies int32[n, trials].  counts: outcome classes 1..6 (PLAYER1 single / gammon /
        backgammon, PLAYER2 the same), truncated trials, plies played."""
        q = _records(positions)
        n, trials = q.shape[0], int(trials)
        o = {"mean": np.zeros(n, np.float64), "std_err": np.zeros(n, np.float64), "counts": np.zeros((n, 8), np.int64)}
        if per_trial:
            o["trial_value"] = np.zeros((n, max(trials, 0)), np.float32)
            o["trial_outcome"] = np.zeros((n, max(trials, 0)), np.int8)
            o["trial_plies"] = np.zeros((n, max(trials, 0)), np.int32)
        L.check(self._lib.bgx_rollout_host(self._h, q.ctypes.data, n, trials, int(max_plies), int(seed) & (2 ** 64 - 1),
                                           L.ROLLOUT_STRATIFY if stratify else 0, L.ptr(o["mean"]), L.ptr(o["std_err"]),
                                           L.ptr(o["counts"]), L.ptr(o.get("trial_value")), L.ptr(o.get("trial_outcome")),
                                           L.ptr(o.get("trial_plies"))))
        return o

    def rollout(self, positions, trials, max_plies=0, seed=0x5EED2026, stratify=True, per_trial=False):
        """rollout_host on a device tensor of positions: the outputs are device tensors, queued on the engine's stream"""
        import torch
        n, trials, dev = positions.shape[0], int(trials), positions.device
        o = {"mean": torch.empty(n, dtype=torch.float64, device=dev), "std_err": torch.empty(n, dtype=torch.float64, device=dev),
             "counts": torch.empty((n, 8), dtype=torch.int64, device=dev)}
        if per_trial:
            o["trial_value"] = torch.empty((n, max(trials, 0)), dtype=torch.float32, device=dev)
            o["trial_outcome"] = torch.empty((n, max(trials, 0)), dtype=torch.int8, device=dev)
            o["trial_plies"] = torch.empty((n, max(trials, 0)), dtype=torch.int32, device=dev)
        L.check(self._lib.bgx_rollout(self._h, L.ptr(positions), n, trials, int(max_plies), int(seed) & (2 ** 64 - 1),
                                      L.ROLLOUT_STRATIFY if stratify else 0, L.ptr(o["mean"]), L.ptr(o["std_err"]),
                                      L.ptr(o["counts"]), L.ptr(o.get("trial_value")), L.ptr(o.get("trial_outcome")),
                                      L.ptr(o.get("trial_plies"))))
        return o

    def twoply_stage_ms(self):
        """Stage times (ms) of the two-ply calls made since the last read with set_option("twoply_timing", 1):
        candidates, expand, replies, reduce"""
        ms = np.zeros(4, np.float64)
        L.check(self._lib.bgx_twoply_stage_ms(self._h, ms.ctypes.data))
        return dict(zip(("candidates", "expand", "replies", "reduce"), ms.tolist()))

    # ------------------------------------------------------------------ self-play population
    def selfplay_init(self, n_slots, first_id=0, id_stride=None, seed=0x5EED2026, first_mover=L.FIRST_ROLLOFF,
                      traj_cap=0, record_chosen=False):
        self.n_slots = int(n_slots)
        self.traj_cap = int(traj_cap)
        self.record_chosen = bool(record_chosen)
        L.check(self._lib.bgx_selfplay_record_chosen(self._h, int(self.record_chosen)))
        L.check(self._lib.bgx_selfplay_init(self._h, int(n_slots), int(first_id), int(id_stride or n_slots),
                                            int(seed), int(first_mover), int(traj_cap)))

    def selfplay_step(self, n_plies, epsilon=0.0, want_stats=True):
        st = L.Stats()
        L.check(self._lib.bgx_selfplay_step(self._h, int(n_plies), float(epsilon), C.byref(st) if want_stats else None))
        return st.as_dict() if want_stats else None

    def selfplay_round(self, epsilon=0.0, want_stats=True):
        st = L.Stats()
        L.check(self._lib.bgx_selfplay_round(self._h, float(epsilon), C.byref(st) if want_stats else None))
        return st.as_dict() if want_stats else None

    def selfplay_next_round(self):
        L.check(self._lib.bgx_selfplay_next_round(self._h))

    def selfplay_read(self):
        rec = np.zeros((self.n_slots, 32), np.int8)
        ply = np.zeros(self.n_slots, np.int32)
        gid = np.zeros(self.n_slots, np.int64)
        L.check(self._lib.bgx_selfplay_read(self._h, rec.ctypes.data, ply.ctypes.data, gid.ctypes.data))
        return rec, ply, gid

    def export_trajectory(self, slot):
        """-> pre int8[T,32] (pre-move records incl. dice), chosen int8[T,32] (afterstates)"""
        cap = max(self.traj_cap, 1)
        pre = np.zeros((cap, 32), np.int8)
        cho = np.zeros((cap, 32), np.int8) if self.record_chosen else None
        T = C.c_int32()
        L.check(self._lib.bgx_export_trajectory(self._h, int(slot), cap, pre.ctypes.data,
                                                cho.ctypes.data if cho is not None else None, C.byref(T)))
        return pre[: T.value], (cho[: T.value] if cho is not None else None)

    def selfplay_sample_host(self, per_game, seed=0):
        """-> int8[n_slots * per_game, 32]: pre-move records of every slot's current game at uniformly drawn plies"""
        out = np.zeros((self.n_slots * int(per_game), 32), np.int8)
        L.check(self._lib.bgx_selfplay_sample_host(self._h, int(per_game), int(seed), out.ctypes.data))
        return out

    def selfplay_sample(self, per_game, seed, out):
        """device tensor int8[n_slots * per_game, 32]"""
        L.check(self._lib.bgx_selfplay_sample(self._h, int(per_game), int(seed), L.ptr(out)))

    # ------------------------------------------------------------------ TD(lambda)
    def td_replay(self, lr, lam, delta, want_stats=True):
        """delta: device fp32[25604] (torch tensor or raw pointer), overwritten with the summed weight change"""
        st = L.Stats()
        L.check(self._lib.bgx_td_replay(self._h, float(lr), float(lam), L.ptr(delta), C.byref(st) if want_stats else None))
        return st.as_dict() if want_stats else None

    def td_replay_scheduled(self, games_done, delta, want_stats=True):
        """td_replay with the reference's per-game lr / lambda schedule (train.py:538, model.py:69-73): the game in global
        slot k of the round is episode games_done + k + 1"""
        st = L.Stats()
        L.check(self._lib.bgx_td_replay_scheduled(self._h, int(games_done), L.ptr(delta), C.byref(st) if want_stats else None))
        return st.as_dict() if want_stats else None

    def apply_delta(self, delta, scale=1.0):
        L.check(self._lib.bgx_apply_delta(self._h, L.ptr(delta), float(scale)))

    def td_profile(self, on=True):
        """Switch the instrumented k_td_replay on/off; -> uint64[8, 16] phase cycles per warp of the last instrumented launch (CTA 0)"""
        out = np.zeros((8, 16), np.uint64)
        L.check(self._lib.bgx_td_profile(self._h, int(bool(on)), out.ctypes.data))
        return out

    def td_replay_host(self, records, player1_won, lr, lam):
        """One trajectory (records int8[T,32], byte 28 = turn flag) from the engine's current weights.
        -> (W1, b1, w2, b2) after the replay, squared TD errors of the T-1 non-terminal steps"""
        r = _records(records)
        T = r.shape[0]
        W1 = np.zeros((128, 198), np.float32)
        b1 = np.zeros(128, np.float32)
        w2 = np.zeros((1, 128), np.float32)
        b2 = np.zeros(1, np.float32)
        sq = np.zeros(max(T - 1, 1), np.float64)
        L.check(self._lib.bgx_td_replay_host(self._h, r.ctypes.data, T, int(bool(player1_won)), float(lr), float(lam),
                                             W1.ctypes.data, b1.ctypes.data, w2.ctypes.data, b2.ctypes.data, sq.ctypes.data))
        return (W1, b1, w2, b2), sq[: max(T - 1, 0)]
