"""Networks served by the caller (c4_net_create_external, connect4_b200/neural/torch_model.py): the device engine keeps the
search, the memo and the records and calls a PyTorch module once per lock-step pass.

(1) A TorchModel that relays to the compiled tower must reproduce the compiled tower's generations and searches bit for
bit; (2) a geometry the library cannot compile runs through ModelWrapper, and its games are replayed by the oracle with
the module's logged answers; (3) the reference-facing surface works on it; (4) failures of the module fail the call and
leave the engine usable."""
from copy import copy

import numpy as np
import pytest

from conftest import GOLDEN, bits, golden, random_positions
from test_torch_net import lively_state

pytestmark = pytest.mark.gpu


def _cfg(sims, alpha=0.3, frac=0.25, sampling=6):
    from connect4_b200.mcts import MCTSConfig
    return MCTSConfig(sims, 19652, 1.25, alpha, frac, sampling)


def _golden_model():
    import os
    from oracle import net_ref as nr
    from connect4_b200.neural.model import ModelWrapper
    return ModelWrapper(state_dict=nr.load_golden_state(os.path.join(GOLDEN, "example_net_state.npz")))


def _relay(mw, state=None):
    """TorchModel whose module sends its planes back to bitboards and through the compiled tower of `mw`: the same numbers
    as the native path, served by the caller.  state["fail"] / state["nan"] / state["shape"] make it misbehave."""
    import torch
    from connect4_b200.board import BoardBatch
    from connect4_b200.neural.torch_model import TorchModel
    state = {} if state is None else state

    def module(planes):
        if state.get("fail"):
            raise RuntimeError("module exploded on purpose")
        bb = BoardBatch.from_planes(planes[:, 1], planes[:, 2])
        v, p = mw.evaluate_bitboards(bb.c0, bb.c1)
        if state.get("nan"):
            v = torch.full_like(v, float("nan"))
        if state.get("shape"):
            p = p[:, :6]
        return v, p
    return TorchModel(module, mw.device)


def _sorted(rec):
    return rec[np.lexsort((rec["ply"], rec["game_id"]))]


def _same(a, b):
    assert len(a) == len(b)
    for f in a.dtype.names:                       # field by field (numpy leaves a record's padding bytes undefined)
        assert a[f].tobytes() == b[f].tobytes(), f


def _generate(monkeypatch, engine, model, cfg, slots, n, seed=3):
    from connect4_b200.neural.game_pool import SelfPlayPool
    if engine is None:
        monkeypatch.delenv("C4_ENGINE", raising=False)
    else:
        monkeypatch.setenv("C4_ENGINE", engine)
    pool = SelfPlayPool(model, cfg, concurrent_games=slots, seed=seed)
    rec = _sorted(pool.generate_records(n))
    pool.engine.close()
    return rec


# ------------------------------------------------------------------------------------------- (1) identity through the new path
@pytest.mark.parametrize("slots,sims,n", [(512, 100, 1024), (4096, 800, 4096)])
def test_relayed_tower_generates_the_native_records(monkeypatch, slots, sims, n):
    """AlphaZero generation (Philox noise, sampled moves), cold memo: records byte-identical to SelfPlayPool(ModelWrapper),
    with the lock-step engine forced and with the default engine (split for the native tower, lock-step for the served one)"""
    mw = _golden_model()
    tm = _relay(mw)
    for engine in ("lockstep", None):
        native = _generate(monkeypatch, engine, mw, _cfg(sims), slots, n)
        served = _generate(monkeypatch, engine, tm, _cfg(sims), slots, n)
        assert sorted(set(served["game_id"].tolist())) == list(range(n))
        _same(native, served)


def test_relayed_tower_search_batch_equals_native():
    from connect4_b200.board import Board
    from connect4_b200.mcts import search_batch
    mw = _golden_model()
    tm = _relay(mw)
    c0, c1 = random_positions(41, 256)
    boards = [Board.from_bitboards(int(a), int(b)) for a, b in zip(c0, c1)]
    cfg = _cfg(200, 0.0, 0.0, 0)
    a = search_batch(cfg, boards, mw).readout(256)
    b = search_batch(cfg, boards, tm).readout(256)
    assert (a["root_visits"] == 201).all()
    for k in ("visits", "best", "nodes", "root_visits"):
        assert (a[k] == b[k]).all(), k
    assert (bits(a["vsum"]) == bits(b["vsum"])).all()


# ------------------------------------------------------------------------------------------- (2) a geometry the library cannot compile
def _net128():
    from connect4_b200.neural.model import ModelWrapper
    sd = lively_state(128, 2, 1)
    return ModelWrapper(state_dict=sd), sd


def test_128_filters_are_served_by_torch_within_the_tolerance():
    from oracle import net_ref as nr
    mw, sd = _net128()
    assert mw.backend == "torch" and mw.flops_per_position > 0
    e = golden("eval_stats.npz")
    v, p = mw.evaluate_bitboards(e["c0"], e["c1"])
    rv, rp = nr.evaluate({k: x.numpy() for k, x in sd.items()}, e["c0"], e["c1"])
    dv, dp = np.abs(v.cpu().numpy() - rv).max(), np.abs(p.cpu().numpy() - rp).max()
    print("128f/2r torch fp16: max|dvalue| %.2e max|dprior| %.2e" % (dv, dp))
    assert rv.std() > 0.003 and rp.std() > 0.01
    assert dv < 1e-2 and dp < 1e-2


def test_128_filter_generation_replayed_by_the_oracle_with_the_logged_answers(oracle):
    """64 AlphaZero games on 64 slots, Philox draws recorded; every answer the module gave is logged by position, and the
    oracle's search fed with those answers and draws plays the same moves with the same values and policies bit for bit"""
    import torch
    from connect4_b200.board import BoardBatch
    from connect4_b200.neural.game_pool import SelfPlayPool
    from connect4_b200.neural.torch_model import TorchModel, TorchNet
    sd = lively_state(128, 2, 1)
    net = TorchNet(sd, torch.float16).to(torch.device("cuda", torch.cuda.current_device()))
    log = {}

    def module(planes):
        v, p = net(planes)
        bb = BoardBatch.from_planes(planes[:, 1], planes[:, 2])
        for a, b, vv, pp in zip(bb.c0.cpu().numpy().view(np.uint64), bb.c1.cpu().numpy().view(np.uint64),
                                v.cpu().numpy(), p.cpu().numpy()):
            log.setdefault((int(a), int(b)), set()).add((float(vv), pp.astype(np.float32).tobytes()))
        return v, p
    sims, G = 64, 64
    pool = SelfPlayPool(TorchModel(module, dtype=torch.float16), _cfg(sims), concurrent_games=G, seed=99)
    pool.engine.set_rng("philox", seed=99, record=True)
    rec = pool.generate_records(G)
    nz, un = pool.engine.recorded_rng()
    pool.engine.close()
    games = {}
    for r in _sorted(rec):
        games.setdefault(int(r["game_id"]), []).append(r)
    assert sorted(games) == list(range(G))

    class Ambiguous(Exception):
        pass

    def ev(a, b):
        answers = log[(int(a), int(b))]
        if len(answers) != 1:        # evaluated twice (memo entry overwritten) with different bits: which one was used?
            raise Ambiguous()
        v, p = next(iter(answers))
        return v, np.frombuffer(p, np.float32).copy()
    replayed = 0
    for gid, recs in games.items():
        try:
            c0 = c1 = 0
            for ply, r in enumerate(recs):
                t = oracle.Tree(oracle.make_config(sims, 19652, 1.25, 0.3, 0.25, 6), c0, c1)
                t.set_noise(nz[gid][ply])
                t.search(ev)
                mv = t.sample_move(un[gid][ply]) if ply < 6 else t.best_move()
                _, _, _, absval = t.root_children()
                assert (int(r["c0"]), int(r["c1"])) == (c0, c1) and int(r["move"]) == mv, (gid, ply)
                assert np.float32(absval[mv]).tobytes() == np.float32(r["search_value"]).tobytes(), (gid, ply)
                assert t.values_policy().astype(np.float32).tobytes() == r["policy"].tobytes(), (gid, ply)
                c0, c1, _ = oracle.drop(c0, c1, mv)
        except Ambiguous:
            continue
        replayed += 1
        if replayed == 4:
            break
    assert replayed == 4


# ------------------------------------------------------------------------------------------- (3) surface
def test_128_filter_model_wrapper_surface():
    import torch
    from connect4_b200.board import Board, BoardBatch
    from connect4_b200.evaluators import Evaluator, evaluate_centre_with_prior
    from connect4_b200.game import Game
    from connect4_b200.match import Match
    from connect4_b200.mcts import MCTS, MCTSConfig
    from connect4_b200.neural.data import Connect4Dataset
    from connect4_b200.neural.game_pool import game_pool
    from connect4_b200.neural.training_game import GameData
    mw, _ = _net128()
    v, p = mw(Board())
    assert v.shape == (1,) and p.shape == (7,) and v.dtype == np.float32 and p.dtype == np.float32
    b2 = Board()
    b2.make_move(3)
    vs, ps = mw([Board(), b2])
    assert vs.shape == (2,) and ps.shape == (2, 7) and abs(float(ps[1].sum()) - 1.0) < 1e-5
    with pytest.raises(TypeError):
        mw("board")
    e = golden("eval_stats.npz")
    planes = BoardBatch(e["c0"], e["c1"]).to_planes("float32").cpu()
    stats = mw.evaluate(Connect4Dataset(planes, torch.as_tensor(e["values"]), torch.as_tensor(e["priors"])), shuffle=False)
    assert 0.0 <= stats.to_dict()["Accuracy"] <= 1.0
    vo = mw.evaluate_value_only(Connect4Dataset(planes, torch.as_tensor(e["values"]), None))
    assert vo.to_dict()["Average loss"] >= 0.0
    # an MCTS player with the bare model plays a Game; a Match against the centre evaluator takes the lock-step path and
    # plays the games of the one-game-at-a-time path
    p1 = MCTS("net128", MCTSConfig(32), mw)
    p2 = MCTS("centre", MCTSConfig(32), Evaluator(evaluate_centre_with_prior))
    assert Game(False, copy(p1), copy(p2), Board()).play() is not None
    match = Match(False, p1, p2, plies=1, switch=True)
    boards = [copy(g._board) for g in match.games]
    res = match.play()
    assert res["wins"] + res["draws"] + res["losses"] == 14
    for i, (g, b) in enumerate(zip(match.games, boards)):
        solo = Game(False, copy(p1), copy(p2), b) if i < match.n else Game(False, copy(p2), copy(p1), b)
        assert solo.play() == g._board.result
        assert solo.move_history.tolist() == g.move_history.tolist(), i
    gd = game_pool(mw, 16, _cfg(32), 16, seed=4)
    assert len(gd) == 16 and all(isinstance(x, GameData) for x in gd)


def test_compiled_geometries_keep_the_cuda_backend():
    from connect4_b200.neural.config import ModelConfig, NetConfig
    from connect4_b200.neural.model import ModelWrapper
    for f in (32, 64):
        assert ModelWrapper(ModelConfig(net_config=NetConfig(filters=f))).backend == "cuda"


# ------------------------------------------------------------------------------------------- (4) failures
def test_module_failures_fail_the_call_and_leave_the_engine_usable(monkeypatch):
    from connect4_b200._lib import C4Error
    from connect4_b200.board import Board
    from connect4_b200.mcts import search_batch
    from connect4_b200.neural.game_pool import SelfPlayPool
    monkeypatch.setenv("C4_ENGINE", "lockstep")
    mw = _golden_model()
    state = {"fail": True}
    tm = _relay(mw, state)
    pool = SelfPlayPool(tm, _cfg(48), concurrent_games=64, seed=8)
    with pytest.raises(C4Error, match="module exploded on purpose") as ei:
        pool.generate_records(64)
    assert isinstance(ei.value.__cause__, RuntimeError) and "caller's evaluator failed" in str(ei.value)
    c0, c1 = random_positions(5, 32)
    boards = [Board.from_bitboards(int(a), int(b)) for a, b in zip(c0, c1)]
    with pytest.raises(C4Error, match="module exploded on purpose"):
        search_batch(_cfg(64, 0.0, 0.0, 0), boards, tm)
    with pytest.raises(C4Error, match="module exploded on purpose"):
        pool.stream(stop_games=8, reset=True, cold_memo=False)
    # the same pool and the same search engine, now with a working module: exactly the native results (nothing of the
    # failed calls -- games left waiting, PENDING memo tags -- leaks into them)
    state["fail"] = False
    _same(_sorted(pool.generate_records(64)), _generate(monkeypatch, "lockstep", mw, _cfg(48), 64, 64, seed=8))
    r = pool.stream(stop_games=8, reset=True)
    assert r["engine"] == "lockstep" and r["games"] >= 8
    a = search_batch(_cfg(64, 0.0, 0.0, 0), boards, tm).readout(32)
    b = search_batch(_cfg(64, 0.0, 0.0, 0), boards, mw).readout(32)
    assert (a["visits"] == b["visits"]).all() and (bits(a["vsum"]) == bits(b["vsum"])).all()
    # non-finite answers and a wrong output shape
    state["nan"] = True
    with pytest.raises(C4Error, match="non-finite"):
        pool.generate_records(64)
    with pytest.raises(C4Error, match="non-finite"):
        search_batch(_cfg(64, 0.0, 0.0, 0), boards, tm)
    state["nan"], state["shape"] = False, True
    with pytest.raises(C4Error, match="expected value"):
        pool.generate_records(64)
    state["shape"] = False
    assert len(pool.generate_records(8)) > 0
    pool.engine.close()


def test_forced_persistent_engines_run_an_external_net_lock_step(monkeypatch):
    mw = _golden_model()
    tm = _relay(mw)
    ref = _generate(monkeypatch, "lockstep", tm, _cfg(64), 200, 320, seed=11)
    for engine in ("split", "fused"):
        _same(ref, _generate(monkeypatch, engine, tm, _cfg(64), 200, 320, seed=11))
        from connect4_b200.neural.game_pool import SelfPlayPool
        pool = SelfPlayPool(tm, _cfg(64), concurrent_games=200, seed=11)
        assert pool.stream(stop_games=20, reset=True, cold_memo=True)["engine"] == "lockstep"
        pool.engine.close()
