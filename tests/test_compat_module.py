"""The drop-in boundary: our `backgammon_env` (pybind11 over the libbgx C-ABI) against a recorded
session of the module, call by call (and against the reference's own module where oracle/_ref holds
a build), and the reference's three pytest tests (pysrc/tests.py)."""
import gzip
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, PKG, golden_weights

OURS = os.path.join(PKG, "lib")
REFDIR = os.path.join(ROOT, "oracle", "_ref")
SCRIPT = os.path.join(ROOT, "tests", "compat_script.py")
TRANSCRIPT = os.path.join(ROOT, "tests", "golden", "compat_transcript.json.gz")


def run_script(module_dir, tmp_path, tag):
    out = tmp_path / f"{tag}.json"
    r = subprocess.run([sys.executable, SCRIPT, module_dir, str(out)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    return json.load(open(out)), r.stdout


def test_transcript_identical_to_recorded_session(tmp_path):
    """Our module's transcript and printed boards against the recorded ones (tests/golden/compat_transcript.json.gz; its
    provenance is in tests/golden/make_compat_transcript.py); a reference build in oracle/_ref, where there is one, is held
    to the same transcript."""
    with gzip.open(TRANSCRIPT, "rt", encoding="utf-8") as f:
        want = json.load(f)
    runs = [run_script(OURS, tmp_path, "ours")]
    if os.path.isdir(REFDIR) and any(f.startswith("backgammon_env") for f in os.listdir(REFDIR)):
        runs.append(run_script(REFDIR, tmp_path, "ref"))
    for got, printed in runs:
        assert len(got) == len(want["transcript"])
        for i, (a, b) in enumerate(zip(got, want["transcript"])):
            assert a == b, (i, a, b)
        assert printed == want["printed"]       # printGameBoard pictures (game.cpp:260-385)


def test_reference_pytests_reexpressed(golden):
    """pysrc/tests.py:12-49 on our module and our TDLGammonModel."""
    import torch
    import bgx  # noqa: F401  (puts the compat module on sys.path)
    import backgammon_env as bg
    from bgx.model import TDLGammonModel
    assert OURS in bg.__file__
    game = bg.Game(0)
    p1, p2 = bg.Player("P1", bg.PlayerType.PLAYER1), bg.Player("P2", bg.PlayerType.PLAYER2)
    game.setPlayers(p1, p2)
    dice = game.roll_dice()
    assert isinstance(game.legalTurnSequences(game.getTurn(), dice[0], dice[1]), list)          # tests.py:12-21
    model = TDLGammonModel()
    g = golden("model.npz")
    W1, b1, w2, b2 = golden_weights(g, "trained")
    sd = {"fc1.weight": torch.from_numpy(W1), "fc1.bias": torch.from_numpy(b1),
          "fc2.weight": torch.from_numpy(w2), "fc2.bias": torch.from_numpy(b2)}
    model.load_state_dict(sd)                                                                    # tests.py:24-31
    game.roll_dice()
    assert isinstance(model.make_move(game, 1), list)                                            # tests.py:34-49
    # the encoder and forward of our model class against the reference's golden outputs
    X = model._encode_states_np(g["states"].astype(np.int64)[g["turn"] == 0], 0)
    assert np.array_equal(X.view(np.uint32), g["X"][g["turn"] == 0].view(np.uint32))
    with torch.inference_mode():
        v = model(torch.from_numpy(g["X"])).squeeze(1).numpy()
    assert np.max(np.abs(v - g["v_trained"]) / np.abs(g["v_trained"])) <= 1e-5


def test_play_game_and_td_updates_compat(golden):
    """The torch restatement of play_game / apply_td_updates (tests/ref_td.py, the checker of the GPU TD tests) keeps
    the reference contract (train.py:64-172) on the compat module and is bit-identical to the reference's own run."""
    import torch
    from bgx.model import TDLGammonModel
    from ref_td import apply_td_updates, play_game
    torch.manual_seed(1)
    m = TDLGammonModel()
    winner, states, total = play_game(m, 1)
    assert winner in (0, 1) and len(states) == total + 1 and states[0].shape == (198,) and states[0].dtype == np.float32
    # TD replay parity with the reference's own apply_td_updates on its golden trajectory
    g, gm = golden("games.npz"), golden("model.npz")
    W1, b1, w2, b2 = golden_weights(gm, "trained")
    m.load_state_dict({"fc1.weight": torch.from_numpy(W1), "fc1.bias": torch.from_numpy(b1),
                       "fc2.weight": torch.from_numpy(w2), "fc2.bias": torch.from_numpy(b2)})
    m.update_learning_params(1)
    for name in m.eligibility_traces:
        m.eligibility_traces[name].zero_()
    enc = [row for row in g["trained5.enc"]]
    losses = apply_td_updates(m, torch.optim.SGD(m.parameters(), lr=0.1), enc, int(g["trained5.winner"]) == 0)
    assert np.allclose(losses, g["trained5.losses"], rtol=1e-6, atol=0)
    for k, name in (("W1", "fc1.weight"), ("b1", "fc1.bias"), ("w2", "fc2.weight"), ("b2", "fc2.bias")):
        assert np.array_equal(m.state_dict()[name].numpy(), g[f"trained5.new_{k}"]), k


def test_checkpoint_discovery_skips_incompatible_files(tmp_path):
    """save_checkpoint writes the reference's 4-tensor state_dict; latest_compatible_model picks the newest file
    that loads into the 198-128-1 net and skips other architectures (train.py:361-381)."""
    import os
    import torch
    from bgx.model import TDLGammonModel
    from bgx.train import latest_compatible_model, model_compatible, save_checkpoint
    assert latest_compatible_model(str(tmp_path / "missing")) is None
    m = TDLGammonModel()
    good = tmp_path / "tdgammon_a.pth"
    save_checkpoint(m, str(good))
    sd = torch.load(str(good), map_location="cpu", weights_only=True)
    assert sorted(sd) == ["fc1.bias", "fc1.weight", "fc2.bias", "fc2.weight"]
    assert sd["fc1.weight"].shape == (128, 198) and sd["fc2.weight"].shape == (1, 128)
    old = tmp_path / "old3layer.pth"                       # the reference's earlier 3-layer checkpoints
    torch.save({"fc1.weight": torch.zeros(80, 198), "fc1.bias": torch.zeros(80), "fc2.weight": torch.zeros(40, 80),
                "fc2.bias": torch.zeros(40), "fc3.weight": torch.zeros(1, 40), "fc3.bias": torch.zeros(1)}, str(old))
    (tmp_path / "notes.txt").write_text("not a checkpoint")
    os.utime(str(good), (1000, 1000))
    os.utime(str(old), (2000, 2000))                       # newer, but incompatible
    assert model_compatible(str(good)) and not model_compatible(str(old))
    assert latest_compatible_model(str(tmp_path)) == "tdgammon_a.pth"
    m2 = TDLGammonModel()
    m2.load_state_dict(sd)
    assert all(torch.equal(a, b) for a, b in zip(m.state_dict().values(), m2.state_dict().values()))


def test_batch_engine_binding_fails_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import bgx  # noqa: F401
    import backgammon_env as bg
    with pytest.raises(RuntimeError) as ei:
        bg.BatchEngine(0)
    assert "no CPU path" in str(ei.value)
