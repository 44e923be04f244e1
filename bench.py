"""bench.py — self-play plies/s of the B200-native engine (BASELINE.json metric), one JSON line.

    python bench.py [--gpus N] [--steps K] [--warmup W]           # our arm
    python bench.py --impl reference [--steps K] [--warmup W]     # the reference's CPU path

Workload (BASELINE.json configs[2]): greedy 1-ply self-play with the 198-128-1 TD-Gammon net,
65,536 concurrent games per GPU, random-init weights (TDLGammonModel() after torch.manual_seed(0)),
epsilon = 0, Philox dice, first mover g % 2, finished games restart in place.  One STEP = every
game of the population plays PLIES_PER_STEP plies (one k_selfplay launch).

  value      plies/s with the population resident in HBM (CUDA events on the launching stream)
  e2e        plies/s through the C-ABI with HOST buffers: every ply the 65,536 (position, dice) records, ply
             numbers and game ids go pinned-host -> device, one iteration of play_game's loop runs for all of
             them (make_move, is_game_over, setTurn, roll_dice: bgx_play_ply_host_async), the next records and
             the winners come back, and the host restarts finished games
  roofline   the self-play kernel against the bound that limits it (warp-instruction issue; the kernel's DRAM traffic
             and the HBM peak beside it), and SURVEY.md §8(d)'s 1,696 B per enumerated afterstate of the
             materialised dataflow as `materialised_equivalent` (DESIGN.md §4)
  cpu_baseline  the reference engine + model.py loop on the host cores (oracle/ref_play.py)
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "backgammon-engine_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

GAMES_PER_GPU = 65536
PLIES_PER_STEP = 16
SEED = 0x5EED2026
BYTES_PER_AFTERSTATE = 1696          # SURVEY.md §8(d): 792 B X written + 792 B X read + 112 B int32[28] row
FLOP_PER_AFTERSTATE = 50944          # dense 198-128-1 forward, as the reference executes it
METRIC = "selfplay_plies_per_sec"
UNIT = "plies/s"


def workload_config(n_gpus):
    return {"workload": "greedy 1-ply self-play, 198-128-1 net random-init (seed 0), eps=0, Philox dice, "
                        "first mover g%2, in-place restart (BASELINE.json configs[2])",
            "games_per_gpu": GAMES_PER_GPU, "plies_per_step": PLIES_PER_STEP, "n_gpus": n_gpus,
            "parallelism": f"games sharded over {n_gpus} GPU(s), no data-path collective; one process per GPU, pinned to the GPU's local CPUs",
            "l2": "256 MiB scratch written between timed steps (L2 flush); population 2 MiB"}


def init_weights():
    """TDLGammonModel() after torch.manual_seed(0): Xavier-uniform gain 0.1, zero biases (model.py:33-61)."""
    import torch
    torch.manual_seed(0)
    fc1 = torch.nn.Linear(198, 128)
    fc2 = torch.nn.Linear(128, 1)
    for m in (fc1, fc2):
        torch.nn.init.xavier_uniform_(m.weight, gain=0.1)
        torch.nn.init.constant_(m.bias, 0)
    return tuple(t.detach().numpy().copy() for t in (fc1.weight, fc1.bias, fc2.weight, fc2.bias))


# ----------------------------------------------------------------------------- reference arm

def peak_json():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0}, "fallback (B200_PROFILING.md)"


def run_reference(args):
    """The reference's own CPU implementation of the path, all host cores, bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import ref_play
    cores = os.cpu_count() or 1
    procs = max(1, min(cores, args.cpu_procs or cores))
    w = init_weights()
    debug_build = None
    # every step is a bounded sample of the workload; the whole run stays within ~3 minutes whatever K is
    args.cpu_seconds = max(1.0, min(args.cpu_seconds, 150.0 / max(args.steps, 1)))
    if ref_play.available():
        kind = "reference"
        for _ in range(args.warmup):
            ref_play.run(w, min(2.0, args.cpu_seconds), procs)
        tot_p = tot_s = tot_t = 0.0
        for _ in range(args.steps):
            r = ref_play.run(w, args.cpu_seconds, procs)
            tot_p += r["plies"]; tot_s += r["sequences"]; tot_t += r["seconds"]
        sample = (f"reference backgammon_env (oracle/_ref, g++ -O2) + {r['model']} make_move loop (numpy encode, torch CPU "
                  f"1 thread/process), {procs} processes x {args.cpu_seconds:g} s per step, greedy self-play from the opening, "
                  "Philox dice of the GPU arm through Game.setDice")
        if ref_play.available(debug=True):           # the build the reference's own makefile ships (makefile:15: Debug), once
            rd = ref_play.run(w, min(3.0, args.cpu_seconds), procs, debug=True)
            debug_build = {"value": rd["plies"] / rd["seconds"], "unit": UNIT, "build": "g++ -O0 -g (CMAKE_BUILD_TYPE=Debug, makefile:15)",
                           "sample": f"{procs} processes x {min(3.0, args.cpu_seconds):g} s"}
    else:
        # the reference did not compile here (no /root/reference at build time): time the oracle port
        kind = "port"
        tot_p, tot_s, tot_t = port_baseline(w, args.cpu_seconds * max(args.steps, 1))
        procs = 1
        sample = f"oracle/bgx_oracle.c greedy self-play, 1 thread, {tot_t:.1f} s"
    value = tot_p / tot_t
    direct = cpp_direct_sample()
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / max(args.steps, 1),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.gpus),
            "sequences_per_sec": tot_s / tot_t,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": procs, "kind": kind, "sample": sample, "enumeration_only": direct,
                             "reference_debug_build": debug_build},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


def cpp_direct_sample(n=1500):
    """SURVEY 8d's C++-direct comparator on ONE core, enumeration only (no Python, no model): the reference's own
    evaluateTurnSequences (oracle/_ref, ~97 % of it mt19937_64 construction in Game::clone) and the oracle port
    (the same algorithm without that cost = the honest CPU ceiling), on the first n positions of the configs[1] sweep."""
    import numpy as np
    from bgx.synth import make_queries
    from oracle.oracle import Oracle, RefHarness
    q, _ = make_queries(n, seed=20260101)
    out = {"positions": n, "cores": 1}
    try:
        orc = Oracle()
        t0 = time.perf_counter()
        ns, _, _ = orc.turn_summary_batch(q, threads=1)
        out["oracle_port_sequences_per_sec"] = float(ns.sum()) / (time.perf_counter() - t0)
        if RefHarness.available():
            ref = RefHarness()
            tot = np.zeros(1, np.int64)
            import ctypes
            secs = ref.lib.ref_bench_enumerate(np.ascontiguousarray(q[:, :28].astype(np.int32)).reshape(-1), np.ascontiguousarray(q[:, 28]),
                                               np.ascontiguousarray(q[:, 29:31]).reshape(-1), n, tot.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)))
            out["reference_sequences_per_sec"] = float(tot[0]) / secs
    except Exception as exc:
        out["error"] = str(exc)
    return out


def port_baseline(w, seconds):
    import numpy as np
    from oracle.oracle import Oracle
    orc = Oracle()
    rng = np.random.default_rng(1)
    from bgx.synth import START_BOARD
    plies = seqs = 0
    t0 = time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        s = np.zeros(28, np.int32)
        s[:24] = START_BOARD
        pl = 0
        while time.perf_counter() - t0 < seconds:
            d1, d2 = (int(x) for x in rng.integers(1, 7, 2))
            idx, after, v, n = orc.greedy_ply(w, s, pl, d1, d2)
            plies += 1
            seqs += n
            if idx >= 0:
                s = after
            if orc.game_over(s) >= 0:
                break
            pl ^= 1
    return plies, seqs, time.perf_counter() - t0


# ----------------------------------------------------------------------------- our arm

def kernel_sass_sha(kernel):
    """sha256 of the SASS of the first function of libbgx.so whose name contains `kernel` (cuobjdump), or None."""
    import hashlib
    import re
    import shutil
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        return None
    try:
        out = subprocess.run([exe, "-sass", os.path.join(PKG, "lib", "libbgx.so")], capture_output=True, text=True, timeout=120).stdout
    except Exception:
        return None
    keep, on = [], False
    for ln in out.splitlines():
        if "Function :" in ln:
            if on:
                break
            on = kernel in ln
        if on:
            keep.append(re.sub(r"/\*[0-9a-f]{4,}\*/", "", ln).strip())     # drop the addresses, keep mnemonics and encodings
    return hashlib.sha256("\n".join(keep).encode()).hexdigest() if keep else None


def capture_facts(name):
    """Numbers of the committed ncu capture of a kernel (profiles/traffic.json) and whether they describe the kernel that is
    loaded: the capture records the sha256 of the kernel's SASS, which must equal that of the library in this tree."""
    try:
        facts = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))[name]
    except Exception as exc:
        return {}, {"verified": False, "why": f"no capture ({exc})"}
    want, got = facts.get("sass_sha256"), kernel_sass_sha(facts.get("sass_function", name))
    if not want or not got:
        return facts, {"verified": False, "why": "no SASS hash in the capture" if not want else f"no function {facts.get('sass_function', name)} in the loaded library (or no cuobjdump)", "file": facts.get("capture")}
    if want != got:
        return facts, {"verified": False, "why": f"SASS hash of the loaded kernel {got[:12]} != capture {want[:12]} (kernel changed since the capture)",
                       "file": facts.get("capture")}
    return facts, {"verified": True, "why": "SASS hash matches", "file": facts.get("capture"), "sass_sha256": got[:16]}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md clocks line)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], threading.Event()

    def run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx[0] if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


def side_legs(eng, dev, peaks, n_positions):
    """The other kernels of the path on BASELINE.json configs[1]'s input (seeded synthetic positions incl. bar
    entry, doubles and bear-off), device-resident, CUDA-event timed inside the library: enumeration only,
    enumeration + evaluation + arg-best, the unfused encoder (the one truly HBM-bound kernel) and the evaluator."""
    import numpy as np
    import torch
    from bgx.synth import make_sweep_queries
    q, _ = make_sweep_queries(eng, n_positions)      # configs[1]: half constructive, half sampled from random playouts
    qd = torch.from_numpy(q).to(dev)
    n = qd.shape[0]
    n_seq = torch.zeros(n, dtype=torch.int32, device=dev)
    n_uni = torch.zeros(n, dtype=torch.int32, device=dev)
    dig = torch.zeros(n, dtype=torch.int64, device=dev)

    def best_ms(fn, reps=3):
        fn()
        ms = []
        for _ in range(reps):
            fn()
            ms.append(eng.last_kernel_ms())
        return min(ms)

    def best_event_ms(fn, reps=3):
        fn()
        ms = []
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ms.append(a.elapsed_time(b))
        return min(ms)

    t_enum = best_ms(lambda: eng.enumerate_summary(qd, n_seq, n_uni, dig)) * 1e-3
    seqs, uniq = int(n_seq.sum().item()), int(n_uni.clamp(min=0).sum().item())
    chosen = torch.zeros((n, 32), dtype=torch.int8, device=dev)
    val = torch.zeros(n, dtype=torch.float32, device=dev)
    t_sel = best_ms(lambda: eng.select_moves(qd, chosen=chosen, value=val)) * 1e-3
    # the materialised list (batched evaluateTurnSequences): every sequence's moves, length and 32-byte state row.
    # Allocation pass (count-only walk + device scan) and write pass, no host round trip between them.
    offs = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    cnt = torch.zeros(n, dtype=torch.int32, device=dev)
    t_cnt = best_event_ms(lambda: eng.enumerate_count(qd, cnt, offs)) * 1e-3
    assert int(offs[-1].item()) == seqs and torch.equal(cnt, n_seq)
    mv = torch.empty((seqs, 8), dtype=torch.int8, device=dev)
    ln = torch.empty(seqs, dtype=torch.int8, device=dev)
    st = torch.empty((seqs, 32), dtype=torch.int8, device=dev)
    t_wr = best_ms(lambda: eng.enumerate(qd, offs, mv, ln, st)) * 1e-3
    del mv, ln, st
    rows = 4 * n
    qrep = qd.repeat(4, 1)
    X = torch.empty((rows, 198), dtype=torch.float32, device=dev)
    t_enc = best_ms(lambda: eng.encode(qrep, X)) * 1e-3
    enc_gbs = rows * (32 + 792) / t_enc / 1e9
    V = torch.zeros(n, dtype=torch.float32, device=dev)
    t_ev = best_ms(lambda: eng.evaluate(qd, V)) * 1e-3
    arena_leg = None
    try:                                             # SURVEY 8(f) row 2: batched head-to-head evaluation (train.py:262-302, benchmark.py:64-130)
        from bgx.evaluate import Arena, RANDOM
        with np.load(os.path.join(ROOT, "tests", "golden", "model.npz")) as z:
            trained = tuple(z[f"trained_{k}"] for k in ("W1", "b1", "w2", "b2"))
        arena = Arena(dev.index or 0)
        games = 4096
        i = np.arange(games)
        arena.play(trained, RANDOM, np.zeros(256, np.int8), np.arange(256) % 2)          # warm-up
        arena_leg = {"games": games}
        for name, opp in (("model_vs_random", RANDOM), ("model_vs_model", init_weights())):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = arena.play(trained, opp, (i % 2).astype(np.int8), i % 2)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            arena_leg[name] = {"seconds": dt, "games_per_sec": games / dt, "plies_per_sec": float(res["plies"].sum()) / dt,
                               "a_win_rate": float(np.mean(res["winner"] == (i % 2)))}
        arena_leg["note"] = ("Arena.play: 4,096 head-to-head games in lockstep, one k_select launch per policy and ply + k_advance; wall clock "
                             "including the host loop.  The reference plays its 2 x 100 evaluation games per checkpoint at ~300 plies/s per core")
        arena.close()
    except Exception as exc:                         # a side figure: never fails the bench
        arena_leg = {"error": str(exc)}
    return {"positions": n, "sequences": seqs, "unique_afterstates": uniq, "arena": arena_leg,
            "enumerate": {"kernel": "k_enumerate_summary", "ms": t_enum * 1e3, "positions_per_sec": n / t_enum,
                          "sequences_per_sec": seqs / t_enum, "unique_afterstates_per_sec": uniq / t_enum},
            "enumerate_materialised": {"kernels": "k_enumerate_count + k_scan_* + k_enumerate_write", "count_and_scan_ms": t_cnt * 1e3,
                                       "write_ms": t_wr * 1e3, "ms": (t_cnt + t_wr) * 1e3, "sequences_per_sec": seqs / (t_cnt + t_wr),
                                       "bytes_written_per_sequence": 41, "write_gbs": seqs * 41 / t_wr / 1e9,
                                       "round1_path_ms": (t_enum + t_wr) * 1e3,
                                       "note": "batched evaluateTurnSequences on device buffers; round 1 ran k_enumerate_summary (exact U + digest) "
                                               "as the allocation pass and scanned on the host (round1_path_ms = summary + write, without its D2H/H2D)"},
            "select": {"kernel": "k_select", "ms": t_sel * 1e3, "positions_per_sec": n / t_sel,
                       "afterstates_enumerated_and_evaluated_per_sec": seqs / t_sel},
            "encode": {"kernel": "k_encode", "rows": rows, "ms": t_enc * 1e3, "rows_per_sec": rows / t_enc,
                       "roofline": {"bound": "hbm", "achieved": enc_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                    "frac": enc_gbs / peaks["hbm_gbs"], "note": "824 B per row: 32 B record read + 792 B fp32[198] written"}},
            "evaluate": {"kernel": "k_evaluate", "ms": t_ev * 1e3, "rows_per_sec": n / t_ev}}


def td_parity(eng):
    """Per-game weight change of k_td_replay against the reference's own apply_td_updates on the 1,024 GPU-exported
    trajectories per weight set of tests/golden/ (td_traj.npz, td_parity.npz; generator: tests/golden/make_golden.py td_parity):
    p50 / p99 / max over the games of max|dw - dw_ref| / max|dw_ref| per tensor.  The engine's weights are replaced."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from conftest import load_golden
    from td_fixture import TdFixture, engine_errors, quantiles
    out = {"metric": "max|dw - dw_ref| / max|dw_ref| per game and tensor, quantiles p50 / p99 / max over 1,024 games",
           "reference": "unmodified apply_td_updates (train.py:124-172), torch CPU fp32, committed as tests/golden/td_parity.npz",
           "fp32_restatement_vs_reference_W1": {"rand": [3.31e-6, 1.07e-5, 1.61e-5], "trained": [1.14e-5, 4.72e-5, 8.39e-5]}}
    for tag in ("rand", "trained"):
        fx = TdFixture(load_golden, tag)
        err, worst, _ = engine_errors(eng, fx)
        out[tag] = {k: list(v) for k, v in quantiles(err).items()}
        out[tag]["worst_step_td_error_diff"] = worst
    return out


def pin_to_gpu_cpus(index):
    """Several ranks on one box: keep this rank's host threads (and its pinned buffers, first-touch) on the CPUs NVML lists as
    local to its GPU, so that the per-ply host<->device traffic of the end-to-end leg does not cross sockets.  Best effort."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


STEP_COUNTS = ("plies", "sequences", "games_finished", "p1_wins", "truncated")


def dump_outputs(out_dir, eng, stats):
    """What the last timed step hands its caller, as .npy files for comparing two builds output for output: the
    population after it (records int8[G,32] -> records.npy float32; ply numbers and game ids -> float64) and the step's
    game counters in STEP_COUNTS order (step_counts.npy float64).  9 MB for one GPU's 65,536 games (rank 0's)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    rec, ply, gid = eng.selfplay_read()
    for name, a in (("records", rec.astype(np.float32)), ("ply", ply.astype(np.float64)), ("game_id", gid.astype(np.float64)),
                    ("step_counts", np.array([stats[k] for k in STEP_COUNTS], np.float64))):
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from bgx.engine import BatchEngine
    from bgx.lib import FIRST_PARITY
    from bgx.synth import START_BOARD

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    numa = pin_to_gpu_cpus(local) if world > 1 else None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    w = init_weights()
    eng = BatchEngine(local)
    if args.selfplay_warps:
        eng.set_option("selfplay_warps", args.selfplay_warps)
    if args.select_warps:
        eng.set_option("select_warps", args.select_warps)
    stream = torch.cuda.current_stream()
    eng.set_stream(stream.cuda_stream)
    eng.set_weights(*w)
    G = GAMES_PER_GPU
    eng.selfplay_init(G, first_id=rank * G, id_stride=world * G, seed=SEED, first_mover=FIRST_PARITY, traj_cap=0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    launches0 = None
    for _ in range(args.warmup):
        eng.selfplay_step(PLIES_PER_STEP, want_stats=False)
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = eng.launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    kernel_ms, plies, seqs, scored, edges = [], 0, 0, 0, 0
    t_wall0 = time.perf_counter()
    for k in range(args.steps):
        flush.fill_(k & 0xFF)                       # L2 flush between timed iterations (not timed)
        ev[k][0].record(stream)
        st = eng.selfplay_step(PLIES_PER_STEP)      # reads the 64-byte stats block back: one sync per step
        ev[k][1].record(stream)
        kernel_ms.append(eng.last_kernel_ms())
        plies += st["plies"]; seqs += st["sequences"]; scored += st["scored"]; edges += st["tree_edges"]
    barrier()
    wall = time.perf_counter() - t_wall0
    launches = eng.launch_count() - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, eng, st)
    step_ms = [a.elapsed_time(b) for a, b in ev]
    total_ms = torch.tensor([sum(step_ms)], dtype=torch.float64, device=dev)
    counts = torch.tensor([plies, seqs, scored], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(counts, op=dist.ReduceOp.SUM)
    total_s = float(total_ms.item()) / 1e3
    plies_all, seqs_all, scored_all = (float(x) for x in counts.tolist())
    value = plies_all / total_s

    # ---- end to end: host-driven self-play through the C-ABI with HOST buffers, one call per ply and part of the
    # population: bgx_play_ply_host_async = one iteration of play_game's loop (train.py:103-121: make_move, is_game_over,
    # setTurn, roll_dice) for a batch of games.  The population is split into three parts, each on its own asynchronous lane
    # (a lane's launch occupies half the SMs, so two are resident at once): while the GPU plays some (H2D of records, next ply
    # numbers and game ids; k_select_order + k_select + k_advance; D2H of the next records and winners) the host handles
    # another (count the ply, restart finished games in place with the next game id).
    e2e_steps = max(2, min(args.steps, 8)) * PLIES_PER_STEP
    from bgx import host as bgx_host
    LANES = args.e2e_lanes
    if args.lane_grid >= 0:
        eng.set_option("select_lane_grid", args.lane_grid)
    pin = lambda shape, dt: torch.zeros(shape, dtype=dt).pin_memory().numpy()
    bufs = [pin((G, 32), torch.int8), pin((G, 32), torch.int8)]
    win = pin((G,), torch.int8)
    h_gid_pin = pin((G,), torch.int64)
    rec, h_ply, h_gid = eng.selfplay_read()          # continue the (desynchronised) games of the population from the host
    h_gid_pin[:] = h_gid
    h_gid = h_gid_pin
    parts = [(i * G // LANES, (i + 1) * G // LANES) for i in range(LANES)]
    cur = [0] * LANES
    stride = world * G
    bufs[0][:] = rec
    bgx_host.advance(bufs[0], bufs[0], SEED, h_ply, h_gid)   # dice of the current ply for every game (undo the flip below)
    bufs[0][:, 28] ^= 1
    bufs[0][:, 31] = 0

    h_ply_pin = pin((G,), torch.int32)
    h_ply_pin[:] = h_ply
    h_ply = h_ply_pin

    def submit(h):                                      # one iteration of play_game's loop for a third of the population
        lo, hi = parts[h]
        eng.play_ply_restart_host_async(h, bufs[cur[h]][lo:hi], h_ply[lo:hi], h_gid[lo:hi], stride, bufs[1 - cur[h]][lo:hi], win[lo:hi],
                                        first_mover=FIRST_PARITY, dice_seed=SEED)

    def advance(h):                                     # nothing per game on the host: finished games restart on the device
        lo, hi = parts[h]
        eng.wait(h)
        cur[h] ^= 1
        return hi - lo

    for h in range(LANES):
        submit(h)
    e2e_plies = 0
    for it in range(-2, e2e_steps):                 # 2 untimed warm-up ply-steps
        if it == 0:
            barrier()                               # drains nothing of ours: the lanes are non-blocking streams
            t0 = time.perf_counter()
        for h in range(LANES):
            n_adv = advance(h)
            submit(h)
            if it >= 0:
                e2e_plies += n_adv
    for h in range(LANES):
        eng.wait(h)
    e2e_s = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_value = e2e_plies * world / float(e2e_s.item())
    sampler.stop_flag.set()
    sampler.join(timeout=3)

    legs = None
    if rank == 0 and args.side_positions > 0:
        legs = side_legs(eng, dev, peak_json()[0], args.side_positions)

    # ---- one TD(lambda) round (BASELINE configs[3]/[4]): play to the end, replay, all-reduce, apply
    td = None
    if args.td_games < 0:                            # BASELINE.json configs[3] / configs[4]
        args.td_games = 262144 if world == 1 else (1 << 20) // world
    if args.td_games > 0:
        from bgx.lib import FIRST_ROLLOFF
        from bgx.parallel import NcclComm, shard
        first, n_slots, stride = shard(args.td_games * world, rank, world)
        eng.selfplay_init(n_slots, first_id=first, id_stride=stride, seed=SEED + 1, first_mover=FIRST_ROLLOFF, traj_cap=2048)
        delta = torch.zeros(25604, dtype=torch.float32, device=dev)
        comm = NcclComm(eng, dist) if world > 1 else None        # the C-ABI's own communicator (bgx_nccl_comm_init)

        def exchange():                                          # bgx_allreduce_delta: ncclAllReduce(sum, fp32[25604]) on the engine's stream
            if comm:
                comm.allreduce_delta(delta)
        exchange()                                               # untimed: NCCL sets the collective up on first use
        barrier()
        td_sampler = ClockSampler(local)                         # every rank watches its own GPU over the round
        td_sampler.start()
        e0, e1, e2, e3 = (torch.cuda.Event(enable_timing=True) for _ in range(4))
        e0.record(stream)
        play = eng.selfplay_round(0.0)
        e1.record(stream)
        tdst = eng.td_replay(0.1, 0.9, delta)
        e2.record(stream)
        exchange()
        reduced = delta.double()
        eng.apply_delta(delta, 1.0 / (args.td_games * world))
        e3.record(stream)
        barrier()
        td_sampler.stop_flag.set()
        td_sampler.join(timeout=3)
        replay_kernel_ms = eng.last_kernel_ms()
        # the collective alone: every rank enters together, 100 back-to-back all-reduces of the 102,416-byte delta
        ar_us = None
        if comm:
            scratch_delta = delta.clone()
            barrier()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record(stream)
            for _ in range(100):
                comm.allreduce_delta(delta)
            a1.record(stream)
            torch.cuda.synchronize()
            ar = torch.tensor([a0.elapsed_time(a1) * 10.0], dtype=torch.float64, device=dev)     # ms / 100 -> us
            dist.all_reduce(ar, op=dist.ReduceOp.MAX)
            ar_us = float(ar.item())
            delta.copy_(scratch_delta)
        # what every rank must agree on: the reduced delta and the weights after the round (SCALE: the same at N = 2, 4, 8 up to
        # the order of the fp32 sums)
        w_after = np.concatenate([np.asarray(a, np.float64).reshape(-1) for a in eng.get_weights()])
        chk = torch.tensor([float(reduced.sum()), float(reduced.abs().sum()), float(w_after.sum()), float(np.abs(w_after).sum())],
                           dtype=torch.float64, device=dev)
        spread = torch.stack([chk, -chk])
        if world > 1:
            dist.all_reduce(spread, op=dist.ReduceOp.MAX)
        spread = (spread[0] + spread[1]).tolist()                # max - min over the ranks: 0 when every rank holds the same bits
        tcl = td_sampler.summary()
        watts = [float(r[2]) for r in td_sampler.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        lo = torch.tensor([-(tcl["sm_mhz"] or 0.0), max(watts) if watts else 0.0, float("sw_power_cap" in tcl["reasons"]),
                           float(bool(set(tcl["reasons"]) - {"sw_power_cap"}))], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(lo, op=dist.ReduceOp.MAX)
        ms = torch.tensor([e0.elapsed_time(e1), e1.elapsed_time(e2), e2.elapsed_time(e3), e0.elapsed_time(e3), replay_kernel_ms], dtype=torch.float64, device=dev)
        cnt = torch.tensor([play["plies"], tdst["td_steps"], play["games_finished"], play["truncated"], tdst["td_live_rows"], tdst["td_lazy_row_steps"]],
                           dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
        ms, cnt = ms.tolist(), cnt.tolist()
        steps_td = max(cnt[1], 1.0)
        # algorithmic work of a TD step as the sparse replay defines it: per live row and hidden unit one trace FMA (+ the
        # gradient product), one weight FMA and the two forward FMAs of the next step = 9 FLOP; per lazily replayed (row, step)
        # a multiply and an FMA = 3 FLOP; ~1,300 FLOP for the hidden / output layer of both states.  Dense, as the reference
        # executes it: ~255 kFLOP per step (SURVEY 8d).
        props_td = eng.device_props()
        fp32_peak_td = world * props_td["sm_count"] * 128 * 2 * peak_json()[0].get("sm_max_mhz", 1965.0) * 1e6 / 1e12   # all ranks
        flop_sparse = (cnt[4] * 9 + cnt[5] * 3) * 128 + steps_td * 1300
        k_s = ms[4] * 1e-3
        tfacts, tstate = capture_facts("k_td_replay")
        td_roof = {"bound": "fp32", "kernel": "k_td_replay", "kernel_ms": ms[4], "unit": "TFLOP/s", "peak": fp32_peak_td,
                   "achieved": flop_sparse / k_s / 1e12, "frac": flop_sparse / k_s / 1e12 / fp32_peak_td,
                   "flop_per_step": flop_sparse / steps_td, "live_rows_per_step": cnt[4] / steps_td, "lazy_row_steps_per_step": cnt[5] / steps_td,
                   "dense_equivalent": {"flop_per_step": 255000, "achieved": steps_td * 255000 / k_s / 1e12,
                                        "ratio": steps_td * 255000 / k_s / 1e12 / fp32_peak_td,
                                        "note": "the reference's dense per-step work (two dense forwards, dense trace and weight update); "
                                                "the kernel touches only live rows, so this is a speed-up over the dense arithmetic"},
                   "capture": tstate,
                   "note": "the step is a chain of dependent phases (first-layer partials -> barrier -> hidden layer -> barrier -> values -> "
                           "row pass), two games per SM; neither FP32 nor memory bounds it (see `issue`), the FLOP figure says how far the "
                           "arithmetic is from mattering"}
        if tfacts.get("warp_inst_per_step") and tstate["verified"]:
            ipk = world * props_td["sm_count"] * 4 * peak_json()[0].get("sm_max_mhz", 1965.0) * 1e6
            td_roof["issue"] = {"unit": "G warp-inst/s", "peak": ipk / 1e9, "achieved": steps_td * tfacts["warp_inst_per_step"] / k_s / 1e9,
                                "frac": steps_td * tfacts["warp_inst_per_step"] / k_s / ipk, "warp_inst_per_step": tfacts["warp_inst_per_step"],
                                "traffic": tfacts.get("dram_bytes_per_launch")}
        td = {"workload": ("TD(lambda) self-play training, 262,144 concurrent games on 1 GPU (BASELINE.json configs[3])" if world == 1 and args.td_games == 262144
                           else f"TD(lambda) self-play training sharded over {world} GPU(s), {args.td_games * world:,} games in total (BASELINE.json configs[4])"
                           if world > 1 and args.td_games * world == 1 << 20 else f"TD(lambda) self-play training, {args.td_games:,} games per GPU"),
              "games": int(args.td_games * world), "plies": int(cnt[0]), "td_steps": int(cnt[1]), "games_finished": int(cnt[2]),
              "truncated": int(cnt[3]), "play_ms": ms[0], "td_replay_ms": ms[1], "allreduce_apply_ms": ms[2], "round_ms": ms[3],
              "plies_per_sec_incl_update": cnt[0] / (ms[3] * 1e-3), "td_steps_per_sec": cnt[1] / (ms[1] * 1e-3),
              "replay_ms_this_rank": e1.elapsed_time(e2),
              "allreduce_us": ar_us,
              "allreduce": "bgx_allreduce_delta (C-ABI, ncclAllReduce sum of fp32[25604] = 102,416 B on a communicator from bgx_nccl_comm_init); "
                           "allreduce_us = mean of 100 back-to-back calls entered together, max over ranks" if comm else None,
              "checksums": {"delta_sum": float(chk[0]), "delta_abs_sum": float(chk[1]), "weights_sum": float(chk[2]), "weights_abs_sum": float(chk[3]),
                            "max_minus_min_over_ranks": spread,
                            "note": "of the all-reduced weight delta and of the weights after the round; identical bits on every rank "
                                    "(max - min = 0), and equal across N = 2, 4, 8 (the same 2^20 games) up to the order of the fp32 sums"},
              "roofline": td_roof,
              "clocks": {"sm_mhz_min_over_ranks": -float(lo[0]), "power_w_max_over_ranks": float(lo[1]),
                         "sw_power_cap_on_some_rank": bool(lo[2] > 0), "other_slowdown_on_some_rank": bool(lo[3] > 0),
                         "samples_rank0": tcl["samples"],
                         "note": "each rank samples its own GPU (nvidia-smi, 0.2 s) over the whole round; median SM clock per rank, min over ranks"},
              "note": "one round: every game played to its end from one snapshot (k_selfplay), exact online TD(lambda) replay "
                      "per game (k_td_replay, lr 0.1, lambda 0.9), all-reduce of fp32[25604], apply; allreduce_apply_ms includes waiting for the "
                      "slowest rank's replay (max over ranks)"}
        if rank == 0 and not args.no_td_parity:
            td["parity"] = td_parity(eng)
        if comm:
            comm.close()

    if rank == 0:
        peaks, peak_src = peak_json()
        facts, facts_state = capture_facts("k_selfplay")
        traffic = facts.get("dram_bytes_per_launch")
        inst_per_ply = facts.get("warp_inst_per_ply")
        k_ms = float(np.mean(kernel_ms))
        seq_per_launch = seqs / args.steps
        scored_per_launch = scored / args.steps
        props = eng.device_props()
        clock_hz = peaks.get("sm_max_mhz", 1965.0) * 1e6
        issue_peak = props["sm_count"] * 4 * clock_hz
        # What bounds the fused ply kernel: warp-instruction issue (integer / branch / shuffle work, 4 schedulers per SM).
        # Instructions per ply come from the committed ncu capture of THIS kernel binary (its SASS hash is checked) and are
        # rescaled by the tree edges per ply counted in this run, so a change of workload mix does not go unnoticed.
        edges_now = edges / max(plies, 1)
        roof = {"bound": "issue", "unit": "G warp-inst/s", "peak": issue_peak / 1e9, "achieved": None, "frac": None,
                "kernel": "k_selfplay", "kernel_ms": k_ms, "traffic": traffic, "capture": facts_state,
                "tree_edges_per_ply": edges_now, "scored_per_ply": scored / max(plies, 1), "peak_source": peak_src}
        if inst_per_ply and facts_state["verified"]:
            scale = edges_now / facts["tree_edges_per_ply"] if facts.get("tree_edges_per_ply") else 1.0
            ach = (plies / args.steps) * inst_per_ply * scale / (k_ms * 1e-3)
            roof.update({"achieved": ach / 1e9, "frac": ach / issue_peak, "warp_inst_per_ply": inst_per_ply * scale,
                         "warp_inst_per_tree_edge": inst_per_ply / facts["tree_edges_per_ply"] if facts.get("tree_edges_per_ply") else None,
                         "note": "warp instructions per ply (smsp__inst_executed.sum of the committed capture / plies of that launch, rescaled "
                                 "by this run's tree edges per ply) x plies/s, against 4 schedulers x SMs x max clock: the share of issue "
                                 "slots the kernel fills.  It is an occupancy of the bound, not proof of minimal work: the work itself is "
                                 "warp_inst_per_tree_edge x tree edges per ply",
                         "pipes_at_capture": {"issue_active_pct": facts.get("issue_active_pct"), **(facts.get("pipe_pct") or {}),
                                              "note": "ncu, same capture: the integer ALU pipe (16 lanes per scheduler, one warp instruction "
                                                      "per 2 cycles) is the busiest unit of the kernel, the FMA pipe is a quarter full"}})
        else:
            print("bench.py: profiles/traffic.json does not describe the k_selfplay in this libbgx.so "
                  f"({facts_state['why']}): roofline.frac is withheld; re-capture with tools/capture_traffic.py", file=sys.stderr)
        if traffic:
            roof["hbm"] = {"achieved": traffic / (k_ms * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                           "frac": traffic / (k_ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                           "note": "the kernel's own DRAM traffic per launch (ncu dram__bytes_read + write): the population is 2 MB and "
                                   "nothing else is read or written; HBM is idle by design"}
        achieved = seq_per_launch * BYTES_PER_AFTERSTATE / (k_ms * 1e-3) / 1e9
        roof["materialised_equivalent"] = {
            "bytes_per_afterstate": BYTES_PER_AFTERSTATE, "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
            "ratio": achieved / peaks["hbm_gbs"],
            "fused_dataflow_bytes_per_afterstate": 32, "fused_dataflow_ratio": seq_per_launch * 32 / (k_ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
            "note": "NOT a utilisation: the bytes SURVEY 8d's materialised dataflow (792 B of features written + 792 B read + "
                    "112 B state row per enumerated afterstate) would move for the sequences this kernel enumerates, over the "
                    "HBM peak; > 1 means no implementation that stages encodings through HBM can keep up.  32 B: one packed "
                    "record per afterstate (fused encode + evaluate); this kernel writes none"}
        fp32_peak = props["sm_count"] * 128 * 2 * clock_hz / 1e12
        fp32_ach = scored_per_launch * FLOP_PER_AFTERSTATE / (k_ms * 1e-3) / 1e12
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": 1e3 * total_s / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": workload_config(world),
                "sequences_per_sec": seqs_all / total_s, "afterstates_scored_per_sec": scored_all / total_s,
                "legal_afterstates_per_sec": seqs_all / total_s,     # BASELINE.json's second metric: every legal turn sequence's afterstate,
                                                                     # enumerated and evaluated (duplicates and twins scored once, counted all)
                "sequences_per_ply": seqs_all / plies_all, "scored_per_ply": scored_all / plies_all,
                "tree_edges_per_ply_rank0": edges / max(plies, 1), "ply_warps_per_cta": eng.kernel_config(),
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": G * 44, "d2h_bytes_per_step": G * 45,
                        "note": "one step = one ply for all 65,536 games through bgx_play_ply_restart_host_async (= make_move + is_game_over + "
                                "setTurn + roll_dice of train.py:103-121 for a batch, finished games restarted in place as train.py:199-220 "
                                "does game after game): three thirds of the population on three lanes of half the SMs each, pinned host "
                                "buffers, H2D (records, ply numbers, game ids) + k_select + D2H (next records, winners, ply numbers, game "
                                f"ids) per ply; the host loop is wait / swap / submit; {e2e_steps} timed ply-steps"},
                "gpu_launches": int(launches),
                "clocks": sampler.summary(),
                "roofline": roof,
                "fp32_dense_equivalent": {"achieved": fp32_ach, "peak": fp32_peak, "unit": "TFLOP/s", "ratio": fp32_ach / fp32_peak,
                                          "note": "afterstates actually scored x 50,944 FLOP of the dense 198-128-1 forward the reference runs; the "
                                                  "kernel evaluates a scored afterstate with 2-4 integer row adds (delta evaluation), so this is a "
                                                  "speed-up over the dense arithmetic, not a pipe utilisation"},
                "wall_s_timed_region": wall}
        if legs:
            line["side_kernels"] = legs
        if td:
            line["td_round"] = td
        if world == 1 and not args.no_cpu_baseline:
            try:
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "1", "--warmup", "0",
                                    "--cpu-seconds", str(args.cpu_seconds)], capture_output=True, text=True, timeout=600)
                ref = json.loads(r.stdout.strip().splitlines()[-1])
                line["cpu_baseline"] = ref["cpu_baseline"]
            except Exception as exc:                 # the baseline is reported, never required
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "reference", "sample": f"failed: {exc}"}
        emit(line)
    eng.close()
    if world > 1:
        dist.destroy_process_group()


def emit(line):
    """The one JSON line goes to the REAL stdout; everything else any library prints (NCCL's version
    banner, warnings) was redirected to stderr at start-up."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU sample length per reference step")
    ap.add_argument("--cpu-procs", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--selfplay-warps", type=int, default=0, help="warps per CTA of k_selfplay (0 = the library's default)")
    ap.add_argument("--select-warps", type=int, default=0, help="warps per CTA of k_select (0 = the library's default)")
    ap.add_argument("--e2e-lanes", type=int, default=3, help="asynchronous lanes of the end-to-end leg (parts of the population in flight)")
    ap.add_argument("--lane-grid", type=int, default=-1, help="CTAs of a lane's launch (-1 = the library's default: half the SMs; 0 = one per SM)")
    ap.add_argument("--side-positions", type=int, default=1000000, help="positions of the enumeration/encode side legs (0 = skip)")
    ap.add_argument("--no-td-parity", action="store_true", help="skip the TD parity block of the td_round object")
    ap.add_argument("--td-games", type=int, default=-1,
                    help="games per GPU in the TD(lambda) round leg (0 = skip; default: 262,144 on one GPU, 2^20 / N on N)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed self-play step computed to DIR/<name>.npy (population and game counters)")
    args = ap.parse_args()
    if args.dump_outputs and args.steps < 1:
        ap.error("--dump-outputs needs --steps >= 1: it writes what the last timed step computed")
    if args.impl == "reference":
        run_reference(args)
    else:
        args.warmup = max(args.warmup, 3)
        run_ours(args)


if __name__ == "__main__":
    main()
