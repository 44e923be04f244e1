"""Rollouts on one GPU (bgx_rollout, DESIGN 7d).

Input: positions drawn by bgx_selfplay_sample from self-play of the trained test net at uniformly drawn plies (one per game).
Measured, each with CUDA events on device buffers after a warm-up call of the same shape:
  * full rollouts (T = 0) of --positions x --trials stratified trials: games/s and plies/s, next to bgx_selfplay_step's plies/s
    (greedy, --slots games) measured in the same process: the rollout walks the same fused greedy ply;
  * the same positions cut at T = 7;
  * the latency of one position x --trials trials;
  * the mean standard error with and without stratification on the same positions and trial counts;
  * plies/s of a quarter of the positions under each warps-per-CTA setting ("rollout_warps").
With --vr-plies V1,V2,... it measures variance-reduced rollouts (bgx_rollout_vr, DESIGN 7e) instead: for each vr_plies (0 is the
plain bgx_rollout) one timed full-game call on the same positions and trials, its wall time, plies/s, expected walks/s, mean squared
standard error, efficiency 1 / (SE^2 x seconds) and the median per-position ratio vr_std_err / std_err.
The card's name and power limit are read in the same run (nvidia-smi, read-only query).

    python tools/rollout_bench.py [--positions 4096] [--trials 1296] [--vr-plies 0,2,8,4096] [--out results.json]
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


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    line = r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown, unknown"
    name, power = (x.strip() for x in line.split(",", 1))
    return {"name": name, "power_limit": power}


def timed(fn, min_s=1.0):
    """-> (ms per call, last result) over a window of at least min_s (CUDA events on the current stream), after one warm-up call"""
    import torch
    fn()
    torch.cuda.synchronize()
    calls, t0 = 0, time.perf_counter()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    while True:
        out = fn()
        calls += 1
        if time.perf_counter() - t0 >= min_s:
            break
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / calls, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--positions", type=int, default=4096)
    ap.add_argument("--trials", type=int, default=1296)
    ap.add_argument("--slots", type=int, default=65536, help="self-play games of the bgx_selfplay_step comparison")
    ap.add_argument("--vr-plies", default=None, help="comma-separated vr_plies values: measure variance-reduced rollouts")
    ap.add_argument("--out", default=None, help="also write the result as JSON to this file")
    a = ap.parse_args()
    import torch
    from conftest import golden_weights, load_golden
    from bgx.engine import BatchEngine
    from bgx.lib import FIRST_PARITY

    if not torch.cuda.is_available():
        raise SystemExit("rollout_bench: no CUDA device")
    res = {"card": card(), "positions": a.positions, "trials": a.trials}
    w = golden_weights(load_golden("model.npz"), "trained")
    eng = BatchEngine(0)
    eng.set_stream(torch.cuda.current_stream().cuda_stream)
    eng.set_weights(*w)
    eng.selfplay_init(a.positions, first_id=0, id_stride=a.positions, seed=20261020, first_mover=FIRST_PARITY, traj_cap=1024)
    eng.selfplay_round(epsilon=0.0)
    pos = eng.selfplay_sample_host(1, seed=20261020)
    pos[:, 29:] = 0
    pd = torch.from_numpy(pos).cuda()
    games = a.positions * a.trials

    def run(p, T=0, stratify=True):
        return lambda: eng.rollout(p, a.trials, max_plies=T, stratify=stratify)

    if a.vr_plies is not None:
        res["vr"] = {v: vr_row(eng, pd, a.trials, int(v)) for v in a.vr_plies.split(",")}
        finish(eng, res, a.out)
        return

    # the self-play reference: greedy bgx_selfplay_step over a population, plies/s
    eng.selfplay_init(a.slots, first_id=0, id_stride=a.slots, seed=7, first_mover=FIRST_PARITY)
    eng.selfplay_step(64)
    torch.cuda.synchronize()
    sp_plies, sp_ms = 0, 0.0
    for _ in range(4):
        st = eng.selfplay_step(64)
        sp_plies += st["plies"]
        sp_ms += eng.last_kernel_ms()
    res["selfplay_step"] = {"slots": a.slots, "plies_per_s": sp_plies / (sp_ms * 1e-3)}
    print(f"selfplay_step: {json.dumps(res['selfplay_step'])}", flush=True)

    for T in (0, 7):
        ms, out = timed(run(pd, T), min_s=0.5)
        plies = int(out["counts"][:, 7].sum().item())
        r = {"ms": ms, "games_per_s": games / (ms * 1e-3), "plies": plies, "plies_per_s": plies / (ms * 1e-3),
             "mean_plies_per_game": plies / games, "truncated": int(out["counts"][:, 6].sum().item())}
        if T == 0:
            r["plies_per_s_vs_selfplay_step"] = r["plies_per_s"] / res["selfplay_step"]["plies_per_s"]
            se_strat = out["std_err"].mean().item()
            _, un = timed(run(pd, 0, stratify=False), min_s=0.0)
            se_plain = un["std_err"].mean().item()
            res["std_err"] = {"stratified_mean": se_strat, "unstratified_mean": se_plain, "ratio": se_strat / se_plain,
                              "note": "the plain formula; with stratification it overestimates the error"}
        res[f"T={T}"] = r
        print(f"T={T}: {json.dumps(r)}", flush=True)
    print(f"std_err: {json.dumps(res['std_err'])}", flush=True)

    one = pd[:1].contiguous()
    ms, out = timed(run(one), min_s=1.0)
    res["one_position"] = {"ms": ms, "plies": int(out["counts"][0, 7].item())}
    print(f"one position: {json.dumps(res['one_position'])}", flush=True)

    quarter = pd[: max(1, a.positions // 4)].contiguous()
    res["warps"] = {}
    for warps in (16, 20, 24, 32):
        eng.set_option("rollout_warps", warps)
        ms, out = timed(run(quarter), min_s=0.0)
        res["warps"][warps] = {"ms": ms, "plies_per_s": int(out["counts"][:, 7].sum().item()) / (ms * 1e-3)}
    eng.set_option("rollout_warps", 20)
    print(f"warps: {json.dumps(res['warps'])}", flush=True)
    finish(eng, res, a.out)


def vr_row(eng, pd, trials, vr):
    """one timed full-game rollout of every position at vr_plies = vr (0: bgx_rollout), with its standard errors"""
    import torch
    ms, out = timed(lambda: eng.rollout(pd, trials, per_trial=True, vr_plies=vr), min_s=0.0)
    plies = out["trial_plies"].to(torch.int64)
    n_plies = int(plies.sum().item())
    se = out["vr_std_err"] if vr else out["std_err"]
    # a VR ply walks the 21 rolls and the roll played, once less when d1 >= d2 (21 of the 36 ordered rolls)
    vr_plies_played = int(plies.clamp(max=vr).sum().item())
    walks = n_plies + (21 - 21 / 36) * vr_plies_played
    mse = float((se ** 2).mean().item())
    r = {"ms": ms, "plies": n_plies, "plies_per_s": n_plies / (ms * 1e-3), "vr_plies_played": vr_plies_played,
         "walks_per_s_expected": walks / (ms * 1e-3), "mean_se": float(se.mean().item()), "mean_se2": mse,
         "efficiency": 1.0 / (mse * ms * 1e-3)}
    if vr:
        live = out["std_err"] > 0                   # a decided position has no variance to reduce
        r["median_se_ratio"] = float((out["vr_std_err"][live] / out["std_err"][live]).median().item())
        r["mean_minus_vr_mean_max_sigma"] = float(((out["mean"] - out["vr_mean"]).abs()[live]
                                                   / (out["std_err"] ** 2 + out["vr_std_err"] ** 2).sqrt()[live]).max().item())
    print(f"vr_plies={vr}: {json.dumps(r)}", flush=True)
    return r


def finish(eng, res, out):
    eng.close()
    print(json.dumps(res))
    if out:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
