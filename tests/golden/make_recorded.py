"""Record, from this project's own code, reference results that the tests compare against when no reference build is
present (oracle/_ref, built by `make -C oracle ref` from the reference's sources, which are not part of this repository).

    python tests/golden/make_recorded.py compat [MODULE_DIR]   # compat_transcript.json.gz: tests/compat_script.py's session
                                                               # (default MODULE_DIR: oracle/_ref, the reference's own module)
    python tests/golden/make_recorded.py fuzz                  # fuzz_summary.npz: C oracle, 4,000 positions
    python tests/golden/make_recorded.py sweep                 # sha256 for tests/test_gpu_parity.py (needs a GPU)

The committed files were recorded with MODULE_DIR = backgammon-engine_b200/lib, the C oracle and the GPU engine.  The last
recorded run against the reference (the round-2 review, VERDICT.md of commit 0f0f152: CPU suite 37 passed with oracle/_ref
present, "transcript identical to the reference module"; GPU suite 47 passed with the harness loaded) found each of them
equal to the reference on exactly these inputs, and backgammon-engine_b200/, include/, oracle/ and tests/ are unchanged
since that run.  Where the reference can be built, the tests compare it live as well, against the same records.
"""
import gzip
import hashlib
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.abspath(os.path.join(HERE, "..", ".."))
sys.path[:0] = [ROOT, os.path.join(ROOT, "backgammon-engine_b200")]

FUZZ_SEED, FUZZ_N = 987654, 4000


def compat(module_dir):
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "transcript.json")
        r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "compat_script.py"), module_dir, path],
                           capture_output=True, text=True, check=True)
        with open(path) as f:
            rec = {"transcript": json.load(f), "printed": r.stdout}
    with gzip.GzipFile(os.path.join(HERE, "compat_transcript.json.gz"), "wb", mtime=0) as f:
        f.write(json.dumps(rec).encode())
    print("compat_transcript.json.gz:", len(rec["transcript"]), "records from", module_dir)


def fuzz():
    """Sequence count and ordered digest (every move, its order and the resulting state) per position."""
    from bgx.synth import make_queries
    from oracle.oracle import Oracle
    q, _ = make_queries(FUZZ_N, seed=FUZZ_SEED)
    n, _, d = Oracle().turn_summary_batch(q)
    np.savez_compressed(os.path.join(HERE, "fuzz_summary.npz"), queries=q, n_seq=n, digest=d)
    print("fuzz_summary.npz:", len(q), "positions,", int(n.sum()), "sequences")


def sweep_sha256(n_seq, digest):
    """Hash of the 10^6-position sweep's counts and digests, as tests/test_gpu_parity.py stores it."""
    return hashlib.sha256(np.ascontiguousarray(n_seq, np.int64).tobytes() + np.ascontiguousarray(digest, np.uint64).tobytes()).hexdigest()


def sweep():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from conftest import golden_weights, load_golden
    from bgx.engine import BatchEngine
    from bgx.synth import make_sweep_queries
    eng = BatchEngine(0)
    eng.set_weights(*golden_weights(load_golden("model.npz"), "rand"))
    q, _ = make_sweep_queries(eng, 1_000_000)
    n, _, d = eng.enumerate_summary_host(q)
    eng.close()
    print("sequences", int(n.sum()), "sha256", sweep_sha256(n, d))


if __name__ == "__main__":
    what = sys.argv[1] if len(sys.argv) > 1 else ""
    if what == "compat":
        compat(os.path.abspath(sys.argv[2] if len(sys.argv) > 2 else os.path.join(ROOT, "oracle", "_ref")))
    elif what == "fuzz":
        fuzz()
    elif what == "sweep":
        sweep()
    else:
        sys.exit(__doc__)
