"""Cost of serving the network from the caller (c4_net_create_external / TorchModel) against the compiled tower.

One cold 4,096-slot, 800-simulation AlphaZero generation per case, the workload of bench.py (`pool.stream(stop_games=4096,
reset=True, cold_memo=True)`, positions/s = root moves played / device time), for
  native 32f          the default network (example_net weights) on the compiled tower, default engine and lock-step
  relay 32f           the same network through a TorchModel whose module relays to the compiled tower
                      (planes -> bitboards -> tower: the same numbers; the difference is the per-pass host round trip)
  native / torch 64f  the example_config shape (64 filters, 6 blocks, 6 fc; seeded init) on the tower and as a TorchNet
  torch 128f          128 filters, 6 blocks, 6 fc (seeded init) through ModelWrapper, which serves it with TorchNet
  layers 64f / 128f   the 64f network above and the torch_128f state dict on the layer-by-layer kernels
                      (ModelWrapper(kernel="layers"), lock-step engine; C4_POOLS=1 / 2 compares one pool with two half pools)
For the lock-step runs the engine's samplers give the passes, the mean tree-pass time and the mean network time, which for
an external network is the synchronise + the callback (c4_ctx_get keys 8-10).  One JSON line per case.

  python tools/external_net_bench.py [--games 4096] [--sims 800] [--out external_net_bench.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    import torch
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:
        pl = "unknown"
    return {"gpu": torch.cuda.get_device_name(0), "power_limit": pl}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=4096)
    ap.add_argument("--sims", type=int, default=800)
    ap.add_argument("--only", default="", help="comma-separated case names")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch
    from connect4_b200.board import BoardBatch
    from connect4_b200.mcts import MCTSConfig
    from connect4_b200.neural.config import ModelConfig, NetConfig
    from connect4_b200.neural.game_pool import SelfPlayPool
    from connect4_b200.neural.model import ModelWrapper, _init_state_dict
    from connect4_b200.neural.torch_model import TorchModel, TorchNet
    from oracle import net_ref as nr
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    head = card()
    print(json.dumps(head), flush=True)
    cfg = MCTSConfig(args.sims, 19652, 1.25, 0.3, 0.25, 6)
    sd32 = nr.load_golden_state(os.path.join(ROOT, "tests", "golden", "example_net_state.npz"))
    mw32 = ModelWrapper(state_dict=sd32)

    def relay(mw):
        def module(planes):
            bb = BoardBatch.from_planes(planes[:, 1], planes[:, 2])
            return mw.evaluate_bitboards(bb.c0, bb.c1)
        return TorchModel(module, dev)

    def net(filters, res, fc):
        torch.manual_seed(0)
        return _init_state_dict(NetConfig(filters=filters, n_fc_layers=fc, n_residuals=res))
    sd64 = net(64, 6, 6)
    mw64 = ModelWrapper(ModelConfig(net_config=NetConfig(filters=64, n_fc_layers=6, n_residuals=6)), state_dict=sd64)
    cases = [
        ("native_32f", lambda: mw32, None),
        ("native_32f_lockstep", lambda: mw32, "lockstep"),
        ("relay_32f", lambda: relay(mw32), None),
        ("native_64f", lambda: mw64, None),
        ("native_64f_lockstep", lambda: mw64, "lockstep"),
        ("torch_64f", lambda: TorchModel(TorchNet(sd64, torch.float16).to(dev), dev, torch.float16), None),
        ("torch_128f", lambda: ModelWrapper(ModelConfig(net_config=NetConfig(filters=128, n_fc_layers=6, n_residuals=6)),
                                            state_dict=net(128, 6, 6)), None),
        ("layers_64f", lambda: ModelWrapper(ModelConfig(net_config=NetConfig(filters=64, n_fc_layers=6, n_residuals=6)),
                                            state_dict=sd64, kernel="layers"), None),
        ("layers_128f", lambda: ModelWrapper(ModelConfig(net_config=NetConfig(filters=128, n_fc_layers=6, n_residuals=6)),
                                             state_dict=net(128, 6, 6), kernel="layers"), None),
    ]
    only = set(filter(None, args.only.split(",")))
    lines = []
    for name, make, engine in cases:
        if only and name not in only:
            continue
        if engine:
            os.environ["C4_ENGINE"] = engine
        else:
            os.environ.pop("C4_ENGINE", None)
        model = make()
        pool = SelfPlayPool(model, cfg, concurrent_games=args.games, seed=0)
        pool.stream(max_ms=300.0, reset=True, cold_memo=True)                # warm-up: modules, cuDNN algorithms
        r = pool.stream(stop_games=args.games, reset=True, cold_memo=True)
        pool.engine.close()
        out = dict(case=name, backend=getattr(model, "backend", "torch"), engine=r["engine"], games=r["games"],
                   positions=r["positions"], device_ms=round(r["device_ms"], 1),
                   positions_per_sec=round(r["positions"] / (r["device_ms"] / 1e3)),
                   evals=r["evals"], memo_hits=r["memo_hits"], passes=r["passes"],
                   tree_ms=round(r["tree_ms"], 4), net_or_callback_ms=round(r["net_ms"], 4),
                   pools=os.environ.get("C4_POOLS", "default"), **head)
        lines.append(out)
        print(json.dumps(out), flush=True)
        del pool, model
        torch.cuda.empty_cache()
    os.environ.pop("C4_ENGINE", None)
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            for ln in [head] + lines:
                f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
