"""Times the UNMODIFIED reference's multiprocess CPU self-play path (TrainingLoop._generate_games,
oinkoink/neural/training.py:99-133: game_pool worker processes x game threads + one InferenceServer process) on the host
cores.  The reference package is imported from baseline/_ref/oinkoink (a git-ignored copy of the unmodified package, put
there by hand) with oracle/ref_shim standing in for the three
uninstalled imports (anytree, matplotlib.pyplot, visdom).  Nothing of this package is on the path.  Prints one JSON line.
Used by bench.py's cpu_baseline leg only (context next to the C port; see DESIGN.md section 5).
usage: run_reference.py --procs P --threads T --games-per-proc N [--sims 800]"""
import argparse
import json
import os
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--procs", type=int, default=max(1, (os.cpu_count() or 2) - 1))
    ap.add_argument("--threads", type=int, default=2)
    ap.add_argument("--games-per-proc", type=int, default=2)
    ap.add_argument("--sims", type=int, default=800)
    a = ap.parse_args()
    ref = os.path.join(HERE, "_ref")
    if not os.path.isdir(os.path.join(ref, "oinkoink")):
        print(json.dumps({"unavailable": "baseline/_ref/oinkoink is absent (copy the unmodified reference package there)"}))
        return
    sys.path.insert(0, os.path.join(ROOT, "oracle", "ref_shim"))
    sys.path.insert(0, ref)
    import torch
    torch.set_num_threads(1)
    from functools import partial
    from multiprocessing import Pipe, Pool
    from oinkoink.mcts import MCTSConfig
    from oinkoink.neural.config import ModelConfig
    from oinkoink.neural.game_pool import game_pool
    from oinkoink.neural.inference_server import InferenceServer
    from oinkoink.neural.pytorch.model import ModelWrapper

    # the reference's own checkpoint and its default network (32f/3r/4fc), CPU inference
    model = ModelWrapper(ModelConfig(use_gpu=False), os.path.join(ref, "oinkoink", "data", "example_net.pth"))
    # TrainingLoop._create_alpha_zero_config(training=True) with AlphaZeroConfig's defaults (neural/config.py:50-67)
    cfg = MCTSConfig(simulations=a.sims, pb_c_base=19652, pb_c_init=1.25, root_dirichlet_alpha=0.3,
                     root_exploration_fraction=0.25, num_sampling_moves=6)
    connections = [[Pipe() for _ in range(a.threads)] for _ in range(a.procs)]
    t0 = time.perf_counter()
    server = InferenceServer(model, [c[1] for sub in connections for c in sub])
    games = []
    with Pool(processes=a.procs) as pool:
        for batch in pool.imap_unordered(partial(game_pool, mcts_config=cfg, n_threads=a.threads, n_games=a.games_per_proc),
                                         connections, chunksize=1):
            games.extend(batch)
    secs = time.perf_counter() - t0
    server.terminate()
    positions = sum(len(g.moves) for g in games)
    print(json.dumps({"positions": positions, "games": len(games), "seconds": secs, "positions_per_sec": positions / secs,
                      "procs": a.procs, "threads": a.threads, "cores": a.procs + 1}), flush=True)


if __name__ == "__main__":
    main()
