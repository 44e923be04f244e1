"""Two-ply move selection on one GPU (bgx_select_moves_2ply, DESIGN 7c).

Input: queries drawn by bgx_selfplay_sample from self-play of the trained test net at uniformly drawn plies.  For K = 0 and
K = 8: queries/s and replies/s over windows of at least one second (CUDA events, device buffers), the stage times of the call
(candidates, expand, replies, reduce: "twoply_timing", which synchronises between stages), and - for K = 0 - a plain
bgx_select_moves launch on the same reply records next to the reply stage.  Then the two-ply vs one-ply Arena win rate of the
same net.  The card's name and power limit are read in the same run (nvidia-smi, read-only query).

    python tools/twoply_bench.py [--queries 65536] [--games 4096] [--out results.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "backgammon-engine_b200"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

ROLLS = [(a, b) for a in range(1, 7) for b in range(1, a + 1)]


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    line = r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown, unknown"
    name, power = (x.strip() for x in line.split(",", 1))
    return {"name": name, "power_limit": power}


def timed(fn, min_s=1.0):
    """-> ms per call over a window of at least min_s (CUDA events on the current stream), after one warm-up call"""
    import torch
    fn()
    torch.cuda.synchronize()
    calls, t0 = 0, time.perf_counter()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    while True:
        fn()
        calls += 1
        if time.perf_counter() - t0 >= min_s:
            break
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / calls


def reply_records(eng, q):
    """The reply records of K = 0, as the library builds them: every distinct afterstate (first appearance) of every query
    without a winning candidate, with the opponent to move, for each of the 21 rolls."""
    off, _, _, st = eng.enumerate_host(q)
    qid = np.repeat(np.arange(len(q)), np.diff(off))
    key = np.concatenate([qid.astype("<i8").view(np.uint8).reshape(-1, 8), st[:, :28].view(np.uint8)], axis=1)
    _, first = np.unique(np.ascontiguousarray(key).view(np.dtype((np.void, 36))).ravel(), return_index=True)
    first = np.sort(first)
    cq, cs = qid[first], st[first]
    p = q[cq, 28].astype(np.int64)
    win = cs[np.arange(len(cs)), 26 + p] == 15
    keep = ~np.isin(cq, np.unique(cq[win]))
    cs = cs[keep]
    rec = np.repeat(cs, len(ROLLS), axis=0)
    rec[:, 28] ^= 1
    rec[:, 29:31] = np.tile(np.array(ROLLS, np.int8), (len(cs), 1))
    rec[:, 31] = 0
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--queries", type=int, default=65536)
    ap.add_argument("--games", type=int, default=4096)
    ap.add_argument("--out", default=None, help="also write the result as JSON to this file")
    a = ap.parse_args()
    import torch
    from conftest import golden_weights, load_golden
    from bgx.engine import BatchEngine
    from bgx.evaluate import Arena, TwoPly
    from bgx.lib import FIRST_PARITY

    if not torch.cuda.is_available():
        raise SystemExit("twoply_bench: no CUDA device")
    res = {"card": card()}
    w = golden_weights(load_golden("model.npz"), "trained")
    eng = BatchEngine(0)
    eng.set_stream(torch.cuda.current_stream().cuda_stream)
    eng.set_weights(*w)
    per = 8
    games = (a.queries + per - 1) // per
    eng.selfplay_init(games, first_id=0, id_stride=games, seed=20261020, first_mover=FIRST_PARITY, traj_cap=1024)
    eng.selfplay_round(epsilon=0.0)
    q = eng.selfplay_sample_host(per, seed=20261020)[: a.queries]
    n = len(q)
    qd = torch.from_numpy(q).cuda()
    outs = {"chosen": torch.empty((n, 32), dtype=torch.int8, device="cuda"), "value": torch.empty(n, dtype=torch.float32, device="cuda"),
            "n_candidates": torch.empty(n, dtype=torch.int32, device="cuda"), "n_expanded": torch.empty(n, dtype=torch.int32, device="cuda")}
    res["queries"] = n
    for K in (0, 8):
        ms = timed(lambda: eng.select_moves_2ply(qd, K, **outs))
        n_rep = int(outs["n_expanded"].sum().item()) * len(ROLLS)
        eng.set_option("twoply_timing", 1)
        eng.twoply_stage_ms()
        reps = 3
        for _ in range(reps):
            eng.select_moves_2ply(qd, K, **outs)
        stages = {k: v / reps for k, v in eng.twoply_stage_ms().items()}
        eng.set_option("twoply_timing", 0)
        r = {"ms_per_call": ms, "queries_per_s": n / (ms * 1e-3), "replies": n_rep, "replies_per_s": n_rep / (ms * 1e-3),
             "candidates": int(outs["n_candidates"].sum().item()), "stage_ms": stages,
             "reply_stage_replies_per_s": n_rep / (stages["replies"] * 1e-3)}
        if K == 0:
            rec = reply_records(eng, q)
            assert len(rec) == n_rep, (len(rec), n_rep)
            rd = torch.from_numpy(rec).cuda()
            val = torch.empty(len(rec), dtype=torch.float32, device="cuda")
            ms1 = timed(lambda: eng.select_moves(rd, value=val))
            r["select_moves_on_reply_records"] = {"ms": ms1, "replies_per_s": len(rec) / (ms1 * 1e-3)}
        res[f"K={K}"] = r
        print(f"K={K}: {json.dumps(r)}", flush=True)
    arena = Arena(0)
    try:
        i = np.arange(a.games)
        side, first = (i % 2).astype(np.int8), ((i // 2) % 2).astype(np.int8)
        for K in (0, 8):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = arena.play(TwoPly(w, K), w, side, first, seed=0x5EED2026)
            dt = time.perf_counter() - t0
            rate = float(np.mean(out["winner"] == side))
            res[f"arena_K={K}"] = {"games": a.games, "win_rate_2ply_vs_1ply": rate, "sigma": 0.5 / np.sqrt(a.games),
                                   "plies": int(out["plies"].sum()), "seconds": dt}
            print(f"arena K={K}: {json.dumps(res[f'arena_K={K}'])}", flush=True)
    finally:
        arena.close()
    eng.close()
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
