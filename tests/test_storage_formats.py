"""On-disk formats of a generation (SURVEY.md 8f-2): games.pkl in the reference's class namespace
(oinkoink/neural/storage.py:12-17) and data.pth (oinkoink/neural/pytorch/data.py:22-33,52-64).
Goldens `games_ref.pkl` / `data_ref.pth` were written by the unmodified reference (tests/golden/generate_goldens.py
storage): two deterministic self-play games (centre evaluator, 30 and 100 simulations)."""
import os
import pickle
import pickletools
import sys

import numpy as np
import pytest

from connect4_b200.board import Board
from connect4_b200.neural.storage import GameStorage, dump_games, load_games
from connect4_b200.neural.training_game import GameData, games_from_records
from connect4_b200.utils import Result

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden")


def test_reference_games_pkl_loads_into_our_classes():
    games = load_games(os.path.join(GOLD, "games_ref.pkl"))
    z = np.load(os.path.join(GOLD, "games.npz"))
    assert [type(g) for g in games] == [GameData, GameData]
    g = games[0]                                          # the 30-simulation game is also stored move by move
    assert g.moves == z["det0_moves"].tolist()
    assert g.result == Result(float(z["det0_result"]))
    assert all(type(b) is Board for b in g.boards)
    assert [int(b.color[0]) for b in g.boards] == z["det0_c0"].astype(np.int64).tolist()
    assert np.array_equal(np.array(g.values), z["det0_values"])
    assert np.array_equal(np.array(g.priors), z["det0_priors"])
    assert g.data.values == [g.result.value] * len(g.moves)


def test_games_pkl_written_here_is_byte_identical_to_the_reference(tmp_path):
    games = load_games(os.path.join(GOLD, "games_ref.pkl"))
    GameStorage().save(games, str(tmp_path))
    ours = open(tmp_path / "games.pkl", "rb").read()
    assert ours == open(os.path.join(GOLD, "games_ref.pkl"), "rb").read()
    names = {a for op, a, _ in pickletools.genops(ours) if isinstance(a, str) and ("oinkoink" in a or "connect4" in a)}
    assert names == {"oinkoink.board", "oinkoink.neural.training_game", "oinkoink.utils"}
    assert not [m for m in sys.modules if m.startswith("oinkoink")]      # the stand-in namespace is gone again


def test_games_from_device_records_round_trip(tmp_path):
    """records (the engine's 64-byte sink format) -> GameData -> games.pkl -> GameData"""
    from connect4_b200.engine import RECORD_DTYPE
    src = load_games(os.path.join(GOLD, "games_ref.pkl"))
    rows = []
    for gid, g in enumerate(src):
        for ply, (b, m, v, p) in enumerate(zip(g.boards, g.moves, g.values, g.priors)):
            r = np.zeros((), RECORD_DTYPE)
            r["c0"], r["c1"] = int(b.color[0]), int(b.color[1])
            r["policy"], r["search_value"], r["result_value"] = p, v, g.result.value
            r["game_id"], r["move"], r["ply"], r["n_moves"] = gid, m, ply, len(g.moves)
            r["result"] = int(g.result.value * 2)
            rows.append(r)
    rec = np.array(rows, RECORD_DTYPE)
    rng = np.random.default_rng(0)
    games = games_from_records(rec[rng.permutation(len(rec))])            # arrival order does not matter
    dump_games(games, str(tmp_path / "g.pkl"))
    back = load_games(str(tmp_path / "g.pkl"))
    for a, b in zip(src, back):
        assert a.moves == b.moves and a.result == b.result
        assert all(x == y for x, y in zip(a.boards, b.boards))
        assert np.allclose(np.array(a.priors), np.array(b.priors), atol=1e-7)     # policies travel as float32
        assert np.allclose(np.array(a.values, float), np.array(b.values, float), atol=1e-7)


@pytest.mark.gpu
def test_data_pth_equals_the_reference_file(tmp_path):
    import torch
    from connect4_b200.neural.data import Connect4Dataset, TrainingDataStorage
    games = load_games(os.path.join(GOLD, "games_ref.pkl"))
    TrainingDataStorage().save(games, str(tmp_path))
    ours = torch.load(str(tmp_path / "data.pth"))
    ref = torch.load(os.path.join(GOLD, "data_ref.pth"))
    assert set(ours) == set(ref) == {"boards", "values", "priors"}
    for k in ref:
        assert ours[k].dtype == ref[k].dtype and ours[k].shape == ref[k].shape, k
        assert torch.equal(ours[k], ref[k]), k
    ds = Connect4Dataset.load(str(tmp_path / "data.pth"))
    assert len(ds) == 2 * sum(len(g.moves) for g in games)
