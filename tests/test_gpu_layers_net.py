"""Kernel "layers" (connect4_b200/csrc/c4_layers.cu): networks of any width on the layer-by-layer tcgen05 kernels.

(1) accuracy against the fp32 restatement on many geometries; (2) the same numbers as the fused tower where both run;
(3) a position's answer is bitwise independent of its batch; (4) the fp16 protection; (5) the engine: oracle replay,
identical records on every lock-step configuration, concurrent engines on one model, the reference surface."""
import os
import threading

import numpy as np
import pytest

from conftest import GOLDEN, golden, random_positions
from test_torch_net import lively_state

pytestmark = pytest.mark.gpu
TOL = 1e-2


def _cfg(sims, alpha=0.3, frac=0.25, sampling=6):
    from connect4_b200.mcts import MCTSConfig
    return MCTSConfig(sims, 19652, 1.25, alpha, frac, sampling)


def _layers(sd, dtype="fp16"):
    from connect4_b200.neural.model import ModelWrapper
    return ModelWrapper(state_dict=sd, kernel="layers", operand_dtype=dtype)


def _reference(sd, c0, c1):
    """the fp32 restatement (oracle/net_ref), on the GPU in true fp32 for large sets"""
    import torch
    from oracle import net_ref as nr
    if len(c0) <= 6000:
        return nr.evaluate({k: (v.numpy() if torch.is_tensor(v) else v) for k, v in sd.items()}, c0, c1)
    tf = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        dsd = {k: torch.as_tensor(np.asarray(v)).cuda() for k, v in sd.items()}
        vs, ps = [], []
        with torch.no_grad():
            for i in range(0, len(c0), 8192):
                v, p = nr.forward_state(dsd, torch.as_tensor(nr.planes_from_bitboards(c0[i:i + 8192], c1[i:i + 8192])).cuda())
                vs.append(v.cpu().numpy())
                ps.append(p.cpu().numpy())
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf
    return np.concatenate(vs), np.concatenate(ps)


def _np(t):
    return t.cpu().numpy()


_BIG = {}


def _big_set():
    """67,557 sampled positions (SURVEY.md 8(d) sampling): more boards than L2 holds activations for at 128 filters"""
    if "c" not in _BIG:
        c0, c1 = random_positions(2024, 67557)
        _BIG["c"] = (np.asarray(c0, np.uint64), np.asarray(c1, np.uint64))
    return _BIG["c"]


# ------------------------------------------------------------------------------------------- (1) accuracy
def test_example_net_golden_fp16_and_bf16():
    from oracle import net_ref as nr
    g = golden("net_outputs.npz")
    sd = nr.load_golden_state(os.path.join(GOLDEN, "example_net_state.npz"))
    m = _layers(sd)
    assert m.backend == "cuda"
    v, p = m.evaluate_bitboards(g["c0"], g["c1"])
    dv, dp = np.abs(_np(v) - g["value"]), np.abs(_np(p) - g["prior"])
    print("example_net layers fp16: max|dvalue| %.2e max|dprior| %.2e" % (dv.max(), dp.max()))
    assert dv.max() < TOL and dp.max() < TOL
    vb, pb = _layers(sd, "bf16").evaluate_bitboards(g["c0"], g["c1"])
    eb = np.abs(_np(vb) - g["value"])
    print("example_net layers bf16: max|dvalue| %.2e mean %.2e" % (eb.max(), eb.mean()))
    assert eb.mean() < 5e-3 and eb.max() < 0.1 and np.abs(_np(pb) - g["prior"]).max() < 0.1


@pytest.mark.parametrize("filters,residuals,fc", [(16, 1, 1), (48, 10, 2), (64, 6, 6), (96, 4, 2), (128, 2, 1),
                                                  (128, 6, 6), (256, 2, 1)])
def test_lively_nets_within_tolerance(filters, residuals, fc):
    from connect4_b200 import _lib
    e = golden("net_outputs.npz")
    sd = lively_state(filters, residuals, fc)
    m = _layers(sd)
    lib = _lib.load()
    assert lib.c4_net_get(m.c4_net, 6) == 2.0 and lib.c4_net_get(m.c4_net, 4) == 0.0 and lib.c4_net_get(m.c4_net, 0) == filters
    v, p = m.evaluate_bitboards(e["c0"], e["c1"])
    rv, rp = _reference(sd, e["c0"], e["c1"])
    dv, dp = np.abs(_np(v) - rv).max(), np.abs(_np(p) - rp).max()
    print("%df/%dr/%dfc layers: max|dvalue| %.2e max|dprior| %.2e (std %.3f %.3f)" % (filters, residuals, fc, dv, dp,
                                                                                       rv.std(), rp.std()))
    assert rv.std() > 0.003 and rp.std() > 0.01                      # the positions really are told apart
    assert dv < TOL and dp < TOL


def test_128_filters_on_67557_positions():
    sd = lively_state(128, 6, 6)
    c0, c1 = _big_set()
    v, p = _layers(sd).evaluate_bitboards(c0, c1)
    rv, rp = _reference(sd, c0, c1)
    dv, dp = np.abs(_np(v) - rv).max(), np.abs(_np(p) - rp).max()
    print("128f/6r/6fc on %d positions: max|dvalue| %.2e max|dprior| %.2e" % (len(c0), dv, dp))
    assert rv.std() > 0.003 and rp.std() > 0.01
    assert dv < TOL and dp < TOL


# ------------------------------------------------------------------------------------------- (2) same numbers as the tower
@pytest.mark.parametrize("filters,residuals,fc", [(32, 3, 4), (64, 6, 6)])
def test_layers_agree_with_the_fused_tower(filters, residuals, fc):
    from connect4_b200 import _lib
    from connect4_b200.neural.model import ModelWrapper
    sd = lively_state(filters, residuals, fc)
    tower, layers = ModelWrapper(state_dict=sd), _layers(sd)
    lib = _lib.load()
    assert (lib.c4_net_get(tower.c4_net, 4), lib.c4_net_get(tower.c4_net, 6)) == (1.0, 1.0)
    assert (lib.c4_net_get(layers.c4_net, 4), lib.c4_net_get(layers.c4_net, 6)) == (0.0, 2.0)
    e = golden("eval_stats.npz")
    v1, p1 = tower.evaluate_bitboards(e["c0"], e["c1"])
    v2, p2 = layers.evaluate_bitboards(e["c0"], e["c1"])
    dv, dp = np.abs(_np(v1) - _np(v2)).max(), np.abs(_np(p1) - _np(p2)).max()
    print("%df tower vs layers: max|dvalue| %.2e max|dprior| %.2e" % (filters, dv, dp))
    assert dv < TOL and dp < TOL


# ------------------------------------------------------------------------------------------- (3) batch independence
def test_answers_are_bitwise_independent_of_the_batch():
    import torch
    from connect4_b200 import _lib
    m = _layers(lively_state(128, 2, 1))
    c0, c1 = _big_set()
    n = len(c0)
    full_v, full_p = m.evaluate_bitboards(c0, c1)
    full = torch.cat([full_p, full_v[:, None]], 1).cpu()
    # shuffled, ragged batches
    perm = np.random.default_rng(5).permutation(n)
    sizes = [1, 2, 127, 129, 4095, 4097, 56, 8191, 16385]
    got = torch.empty_like(full)
    i = k = 0
    while i < n:
        idx = perm[i:i + sizes[k % len(sizes)]]
        v, p = m.evaluate_bitboards(c0[idx], c1[idx])
        got[torch.as_tensor(idx)] = torch.cat([p, v[:, None]], 1).cpu()
        i += len(idx)
        k += 1
    assert torch.equal(got, full)
    # a device count smaller than n: rows past it untouched
    t0 = torch.as_tensor(c0[:20000].view(np.int64)).cuda()
    t1 = torch.as_tensor(c1[:20000].view(np.int64)).cuda()
    out = torch.full((20000, 8), -7.0, dtype=torch.float32, device="cuda")
    cnt = torch.tensor([12345], dtype=torch.int32, device="cuda")
    _lib.check(_lib.load().c4_net_forward(m.c4_net, _lib.ptr(t0), _lib.ptr(t1), 20000, _lib.ptr(cnt), _lib.ptr(out),
                                          _lib.stream_ptr()))
    torch.cuda.synchronize()
    assert torch.equal(out[:12345].cpu(), full[:12345]) and (out[12345:] == -7.0).all()
    v, p = m.evaluate_bitboards(np.zeros(0, np.uint64), np.zeros(0, np.uint64))
    assert v.numel() == 0 and p.shape == (0, 7)


# ------------------------------------------------------------------------------------------- (4) fp16 safety
def test_fp16_trunk_scale_and_nan_refusal():
    import torch
    from connect4_b200._lib import C4Error
    from connect4_b200.neural.game_pool import SelfPlayPool
    from oracle import net_ref as nr
    from test_gpu_net import _scaled_trunk_state
    sd = _scaled_trunk_state(3.0e5)
    g = golden("net_outputs.npz")
    rv, rp = nr.evaluate(sd, g["c0"], g["c1"])
    m = _layers(sd)
    assert m.trunk_scale_log2 >= 8
    v, p = m.evaluate_bitboards(g["c0"], g["c1"])
    assert np.isfinite(_np(v)).all()
    assert np.abs(_np(v) - rv).max() < TOL and np.abs(_np(p) - rp).max() < TOL
    sd = {k: torch.as_tensor(np.array(x)).clone() for k, x in nr.load_golden_state(os.path.join(GOLDEN, "example_net_state.npz")).items()}
    sd["policy_head.fc1.weight"][3, 5] = float("nan")
    pool = SelfPlayPool(_layers(sd), _cfg(16), concurrent_games=4, seed=1)
    with pytest.raises(C4Error, match="non-finite"):
        pool.generate_records(4)
    pool.engine.close()
    sd["body.0.0.weight"][0, 0, 0, 0] = float("nan")                 # NaN in the trunk: refused at creation
    with pytest.raises(C4Error):
        _layers(sd)


# ------------------------------------------------------------------------------------------- (5) engine
_M128 = {}


def _net128():
    if "m" not in _M128:
        _M128["m"] = _layers(lively_state(128, 2, 1))
    return _M128["m"]


def _sorted(rec):
    return rec[np.lexsort((rec["ply"], rec["game_id"]))]


def _same(a, b):
    assert len(a) == len(b)
    for f in a.dtype.names:
        assert a[f].tobytes() == b[f].tobytes(), f


def _generate(monkeypatch, model, slots, sims, n, env=(), seed=3):
    from connect4_b200.neural.game_pool import SelfPlayPool
    for k in ("C4_ENGINE", "C4_POOLS", "C4_NO_GRAPH"):
        monkeypatch.delenv(k, raising=False)
    for k, v in env:
        monkeypatch.setenv(k, v)
    pool = SelfPlayPool(model, _cfg(sims), concurrent_games=slots, seed=seed)
    rec = _sorted(pool.generate_records(n))
    info = pool.engine
    pool.engine.close()
    for k, _ in env:
        monkeypatch.delenv(k, raising=False)
    return rec, info


def test_generation_replayed_bit_for_bit_by_the_oracle(oracle):
    from connect4_b200.neural.game_pool import SelfPlayPool
    m = _net128()
    sims, G = 64, 64
    pool = SelfPlayPool(m, _cfg(sims), concurrent_games=G, seed=99)
    pool.engine.set_rng("philox", seed=99, record=True)
    rec = pool.generate_records(G)
    nz, un = pool.engine.recorded_rng()
    pool.engine.close()
    games = {}
    for r in _sorted(rec):
        games.setdefault(int(r["game_id"]), []).append(r)
    assert sorted(games) == list(range(G))
    cache = {}

    def ev(a, b):                           # the same model on the one position: batch independence makes it exact
        key = (int(a), int(b))
        if key not in cache:
            v, p = m.evaluate_bitboards(np.array([a], np.uint64), np.array([b], np.uint64))
            cache[key] = (float(_np(v)[0]), _np(p)[0].astype(np.float32))
        v, p = cache[key]
        return v, p.copy()
    for gid in range(8):
        c0 = c1 = 0
        for ply, r in enumerate(games[gid]):
            t = oracle.Tree(oracle.make_config(sims, 19652, 1.25, 0.3, 0.25, 6), c0, c1)
            t.set_noise(nz[gid][ply])
            t.search(ev)
            mv = t.sample_move(un[gid][ply]) if ply < 6 else t.best_move()
            _, _, _, absval = t.root_children()
            assert (int(r["c0"]), int(r["c1"])) == (c0, c1) and int(r["move"]) == mv, (gid, ply)
            assert np.float32(absval[mv]).tobytes() == np.float32(r["search_value"]).tobytes(), (gid, ply)
            assert t.values_policy().astype(np.float32).tobytes() == r["policy"].tobytes(), (gid, ply)
            c0, c1, _ = oracle.drop(c0, c1, mv)


def test_records_identical_on_every_lockstep_configuration(monkeypatch):
    m = _net128()
    base, _ = _generate(monkeypatch, m, 512, 100, 1024)
    assert sorted(set(base["game_id"].tolist())) == list(range(1024))
    for env in ((("C4_NO_GRAPH", "1"),), (("C4_POOLS", "1"),), (("C4_POOLS", "2"),), (("C4_ENGINE", "split"),)):
        rec, _ = _generate(monkeypatch, m, 512, 100, 1024, env)
        _same(base, rec)


def test_split_engine_falls_back_to_lockstep(monkeypatch):
    from connect4_b200.neural.game_pool import SelfPlayPool
    monkeypatch.setenv("C4_ENGINE", "split")
    pool = SelfPlayPool(_net128(), _cfg(50), concurrent_games=64, seed=1)
    r = pool.stream(stop_games=64, reset=True)
    pool.engine.close()
    assert r["engine"] == "lockstep"


@pytest.mark.parametrize("slots,sims,n", [(512, 100, 1024), (4096, 800, 4096)])
def test_relayed_layers_give_the_native_records(monkeypatch, slots, sims, n):
    from connect4_b200.board import BoardBatch
    from connect4_b200.neural.torch_model import TorchModel
    m = _net128()

    def module(planes):
        bb = BoardBatch.from_planes(planes[:, 1], planes[:, 2])
        return m.evaluate_bitboards(bb.c0, bb.c1)
    native, _ = _generate(monkeypatch, m, slots, sims, n)
    served, _ = _generate(monkeypatch, TorchModel(module, m.device), slots, sims, n)
    assert sorted(set(served["game_id"].tolist())) == list(range(n))
    _same(native, served)


def test_two_engines_share_one_model_concurrently(monkeypatch):
    import torch
    from connect4_b200.neural.game_pool import SelfPlayPool
    for k in ("C4_ENGINE", "C4_POOLS", "C4_NO_GRAPH"):
        monkeypatch.delenv(k, raising=False)
    m = _net128()
    seeds = (11, 12)
    alone = [_generate(monkeypatch, m, 256, 100, 512, seed=s)[0] for s in seeds]
    pools = [SelfPlayPool(m, _cfg(100), concurrent_games=256, seed=s) for s in seeds]
    out, errors = [None, None], []

    def run(i):
        try:
            with torch.cuda.stream(torch.cuda.Stream()):
                out[i] = _sorted(pools[i].generate_records(512))
                torch.cuda.current_stream().synchronize()
        except Exception as e:            # (re-raised below, on the test's thread)
            errors.append(e)
    th = [threading.Thread(target=run, args=(i,)) for i in range(2)]
    for t in th:
        t.start()
    # meanwhile, public forwards of the same model on the main thread's stream
    c0, c1 = random_positions(8, 3000)
    c0, c1 = np.asarray(c0, np.uint64), np.asarray(c1, np.uint64)
    ref_v, _ = m.evaluate_bitboards(c0, c1)
    ref_v = _np(ref_v)
    while any(t.is_alive() for t in th):
        v, _ = m.evaluate_bitboards(c0, c1)
        assert (_np(v) == ref_v).all()
    for t in th:
        t.join()
    for p in pools:
        p.engine.close()
    assert not errors, errors
    for i in range(2):
        _same(alone[i], out[i])


def test_reference_surface():
    from copy import copy
    from connect4_b200.board import Board
    from connect4_b200.evaluators import Evaluator, evaluate_centre_with_prior
    from connect4_b200.game import Game
    from connect4_b200.match import Match
    from connect4_b200.mcts import MCTS, MCTSConfig, search_batch
    m = _net128()
    assert m.backend == "cuda" and m.flops_per_position > 0
    v, p = m(Board())
    assert v.shape == (1,) and p.shape == (7,) and v.dtype == np.float32
    b2 = Board()
    b2.make_move(3)
    vs, ps = m([Board(), b2])
    assert vs.shape == (2,) and ps.shape == (2, 7) and abs(float(ps[1].sum()) - 1.0) < 1e-5
    assert vs[0] == v[0] and (ps[0] == p).all()
    c0, c1 = random_positions(41, 64)
    boards = [Board.from_bitboards(int(a), int(b)) for a, b in zip(c0, c1)]
    out = search_batch(_cfg(100, 0.0, 0.0, 0), boards, m).readout(64)
    assert (out["root_visits"] == 101).all()
    p1 = MCTS("layers128", MCTSConfig(32), m)
    p2 = MCTS("centre", MCTSConfig(32), Evaluator(evaluate_centre_with_prior))
    assert Game(False, copy(p1), copy(p2), Board()).play() is not None
    res = Match(False, p1, p2, plies=1, switch=True).play()
    assert res["wins"] + res["draws"] + res["losses"] == 14
