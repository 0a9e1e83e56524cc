"""Stand-alone forward of the layer-by-layer network kernels (kernel "layers", connect4_b200/csrc/c4_layers.cu) against
the fused tcgen05 tower where it exists (64 filters), timed with CUDA events.

For each network and batch size: warm-up, then `--reps` back-to-back forwards between two events; TFLOP/s = algorithmic
FLOPs (c4_net_flops_per_position x positions) over the mean time per forward.  Inputs: sampled positions (random stones,
0..34 plies).  Working sets: at 67,557 positions the activations (56 rows x (4 + 2 + 2) bytes x F per position) exceed the
126 MB L2 from 64 filters up; the smaller batches run L2-resident, as in self-play.  One JSON line per (network, batch).

  python tools/layers_time.py [--reps 20] [--out profiles/layers_forward.jsonl]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import numpy as np
    import torch
    from connect4_b200 import _lib
    from connect4_b200.neural.config import NetConfig
    from connect4_b200.neural.model import ModelWrapper, _init_state_dict
    from external_net_bench import card
    torch.cuda.set_device(0)
    head = card()
    print(json.dumps(head), flush=True)
    rng = np.random.default_rng(0)
    N = 67557
    c0 = np.zeros(N, np.uint64)
    c1 = np.zeros(N, np.uint64)
    for i in range(N):                     # random legal-shaped positions: column heights, alternate colours
        h = [0] * 7
        for k in range(int(rng.integers(0, 35))):
            col = int(rng.integers(0, 7))
            if h[col] == 6:
                continue
            bit = np.uint64(1 << (7 * col + h[col]))
            h[col] += 1
            if k & 1:
                c1[i] |= bit
            else:
                c0[i] |= bit
    t0 = torch.as_tensor(c0.view(np.int64)).cuda()
    t1 = torch.as_tensor(c1.view(np.int64)).cuda()
    out = torch.empty((N, 8), dtype=torch.float32, device="cuda")
    lib = _lib.load()
    lines = []
    for filters, res, fc, kernel in [(64, 6, 6, "auto"), (64, 6, 6, "layers"), (128, 6, 6, "layers"), (256, 6, 6, "layers")]:
        torch.manual_seed(0)
        sd = _init_state_dict(NetConfig(filters=filters, n_fc_layers=fc, n_residuals=res))
        m = ModelWrapper(state_dict=sd, kernel=kernel)
        which = {0: "mma.sync", 1: "tower", 2: "layers"}[int(lib.c4_net_get(m.c4_net, 6))]
        flops = m.flops_per_position
        for n in (148, 1184, 2400, 4096, 16384, 67557):
            def fwd():
                _lib.check(lib.c4_net_forward(m.c4_net, _lib.ptr(t0), _lib.ptr(t1), n, None, _lib.ptr(out), _lib.stream_ptr()))
            for _ in range(3):
                fwd()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.reps):
                fwd()
            e1.record()
            e1.synchronize()
            ms = e0.elapsed_time(e1) / args.reps
            ln = dict(net="%df/%dr/%dfc" % (filters, res, fc), kernel=which, positions=n, ms=round(ms, 4),
                      tflops=round(flops * n / (ms * 1e-3) / 1e12, 1), **head)
            lines.append(ln)
            print(json.dumps(ln), flush=True)
        del m
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            for ln in [head] + lines:
                f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
