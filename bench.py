#!/usr/bin/env python3
"""bench.py -- self-play positions/sec at 800 sims/move (BASELINE.json metric) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--engine auto|split|fused|lockstep]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

Workload (ours): BASELINE.json configs[2] as SURVEY.md 8(d) defines it -- 4096 concurrent self-play games per GPU from
the empty board, default NetConfig ResNet (32 filters / 3 residual / 4 fc; the reference's example_net weights), 800
simulations per move, AlphaZero root noise + 6 sampled moves, finished games re-seeded at once, run until 4096 games
have completed -- FROM A COLD EVALUATION MEMO (the reference's position_table lives for one generation,
oinkoink/neural/game_pool.py:21-27).  Games never interact, so with N GPUs every rank runs its own pool (weak scaling).

A "step" = one such generation: fresh pool, empty memo, until `--games` games have finished.
  value = positions (root moves played) of all ranks / device time (CUDA events, max over ranks), inputs resident.
  e2e   = the same metric through the public API with HOST buffers: a whole generation of `--e2e-games` games per GPU
          (4 pool-fulls, drain of the last games included) from pinned host start positions to host records, memo
          cold; with N > 1 through dist.generate_sharded(dst=0), i.e. the NCCL all-gather of every rank's records, the
          device-side sort and the copy of the whole generation to rank 0's host are inside the timed region.
  generation_1200 = BASELINE.json configs[3]: the reference's example_config generation (1200 games, 64f/6r/6fc
          network) sharded over the N GPUs incl. the all-gather; seconds and the digest of the gathered records
          (identical for every N).
  steady_state = the warm regime (memo filled by several seconds of play) -- context only, a real generation never
          gets there.
  roofline = the engine's dominant kernel.  Split engine (default): ONE persistent launch per step (k_sp_one) whose CTAs
          take a role by index -- tree CTAs (HBM class: 1.28 KB per simulation + 64 B per memo probe, SURVEY.md 8d; they
          bound the step and are `roofline`) and tower CTAs (tensor: network FLOPs / step time vs the measured sustained
          bf16 peak; `roofline_other`).  Fused engine: ONE kernel (k_fused) holds both roles; its tensor-side
          figure is `roofline`, its HBM-side figure `roofline_other`.  Lock-step engine: the tree pass / the network
          kernel from launch durations sampled with CUDA events.
          `traffic` = DRAM bytes per launch from the committed ncu capture of the same command and launch shape
          (profiles/r02_split_adapt_launches.csv; split engine, default workload), else null: no DRAM counter is read inside a run.
  cpu_baseline = the oracle port (oracle/selfplay_port.py) on the box's host cores, bounded sample (rank 0, N=1 only).
  cpu_baseline_reference = the unmodified reference package (baseline/_ref, a git-ignored copy put there by hand; reported
          as unavailable without it) on the same cores: its multiprocess game_pool + InferenceServer path, a bounded sample of
          whole games -- context for how conservative the port is.
--impl reference: the CPU port alone, all host cores, same metric / config.
--dump-outputs DIR: after the timed steps, DIR/<name>.npy (float64 / float32) holds what a caller received from them:
  step_{positions,games,evals,memo_hits} = the counters of the last timed step (rank 0; they depend on where the stop lands,
  so they vary slightly from run to run), and records_<field> = the position records of the timed end-to-end generation
  (unless --no-e2e), sorted by game and ply; a seeded sample of rows keeps the whole dump under 64 MB.  The inputs are
  seeded, so two builds run with the same arguments can be compared array by array.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "selfplay_positions_per_sec_at_800_sims_per_move"
UNIT = "positions/s"
SIMS = 800
STATE = os.path.join(ROOT, "tests", "golden", "example_net_state.npz")
WORKLOAD = ("BASELINE.json configs[2]: 4096 concurrent self-play games per GPU, default NetConfig 32f/3r/4fc "
            "(example_net weights), 800 sims/move, AlphaZero noise alpha=0.3 frac=0.25, 6 sampled moves, 16-bit (fp16 operand / fp32 accumulate) tensor-core leaf eval")
DUMP_BYTES = 63 << 20                                   # --dump-outputs: record columns; with the rest under 64 MB


def peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["bf16_tflops_sustained"]), float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json, sustained bf16)"
    except Exception:
        return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region"""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_port(seconds, warm=2.0, procs=None):
    from oracle.selfplay_port import PortPool
    pp = PortPool(procs, SIMS, games_per_worker=32, state_path=STATE)
    try:
        pp.step(warm)
        r = pp.step(seconds)
    finally:
        pp.close()
    return r, pp.procs


def reference_python(timeout_s=240):
    """second stated CPU baseline: the UNMODIFIED reference's multiprocess self-play (TrainingLoop._generate_games,
    oinkoink/neural/training.py:99-133) from baseline/_ref on the host cores, CPU inference, a bounded sample of whole games"""
    procs = max(1, (os.cpu_count() or 2) - 1)                              # + the InferenceServer process = all cores
    cmd = [sys.executable, os.path.join(ROOT, "baseline", "run_reference.py"), "--procs", str(procs), "--threads", "2",
           "--games-per-proc", "2", "--sims", str(SIMS)]
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", OMP_NUM_THREADS="1")
    try:
        out = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=timeout_s).stdout
        r = json.loads([l for l in out.splitlines() if l.startswith("{")][-1])
    except Exception as e:                                                 # context only: never fails the bench line
        return {"unavailable": "%s: %s" % (type(e).__name__, str(e)[:120])}
    if "unavailable" in r:
        return r
    return {"value": r["positions_per_sec"], "unit": UNIT, "cores": r["cores"], "kind": "reference",
            "sample": "unmodified reference package (baseline/_ref), its own checkpoint example_net.pth on CPU: %d game_pool "
                      "processes x %d game threads + 1 InferenceServer process, %d whole games (%d positions) at %d sims/move "
                      "in %.1f s" % (r["procs"], r["threads"], r["games"], r["positions"], SIMS, r["seconds"])}


def run_reference(args, rank):
    """the reference arm: the CPU port of the reference path on all host cores (the reference itself is pure Python
    and is not present on the GPU box; see DESIGN.md)."""
    if rank != 0:
        return
    from oracle.selfplay_port import PortPool
    procs = os.cpu_count() or 1
    pp = PortPool(procs, SIMS, games_per_worker=32, state_path=STATE)
    try:
        budget = args.ref_seconds
        for _ in range(args.warmup):
            pp.step(min(budget, 3.0))
        pos = secs = evals = 0
        for _ in range(args.steps):
            r = pp.step(budget)
            pos += r["positions"]
            secs += r["seconds"]
            evals += r["evals"]
    finally:
        pp.close()
    v = pos / secs
    sample = ("%d single-threaded workers x 32 games in flight, %d steps x %.0f s of self-play at 800 sims/move (C oracle "
              "tree + torch fp32 net + per-process evaluation memo like Evaluator.position_table)" % (
                  procs, args.steps, budget))
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000.0 * secs / max(args.steps, 1), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "host": "CPU port of the reference path (oracle/selfplay_port.py)"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": procs, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "evals_per_sec": evals / secs, "gpu_launches": 0}), flush=True)


def digest_records(rec):
    import hashlib
    import numpy as np
    h = hashlib.sha256()                   # field by field: numpy leaves the 4 padding bytes of a record undefined
    for f in rec.dtype.names:
        h.update(np.ascontiguousarray(rec[f]).tobytes())
    return h.hexdigest()[:16]


def dump_outputs(path, step, rec):
    """--dump-outputs: the last timed step's counters and the end-to-end generation's records (or None) as .npy files"""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    out = {"step_" + k: np.array([step[k]], np.float64) for k in ("positions", "games", "evals", "memo_hits")}
    if rec is not None:
        rec = rec[np.lexsort((rec["ply"], rec["game_id"]))]          # the engine writes records in the order games finish
        cols = {"records_" + f: rec[f].astype(np.float64) for f in ("c0", "c1", "game_id", "move", "ply", "n_moves", "result")}
        cols.update({"records_" + f: rec[f].astype(np.float32) for f in ("policy", "result_value", "search_value")})
        row_bytes = sum(a.nbytes for a in cols.values()) // max(1, len(rec))
        if len(rec) * row_bytes > DUMP_BYTES:
            keep = np.sort(np.random.default_rng(0).choice(len(rec), DUMP_BYTES // row_bytes, replace=False))
            cols = {k: a[keep] for k, a in cols.items()}
        out.update(cols)
    for k, a in out.items():
        np.save(os.path.join(path, k + ".npy"), a)


def ncu_traffic(path, kernel="k_sp_one"):
    """mean over the launches of `kernel` in an ncu --csv metrics file of dram__bytes_read.sum + dram__bytes_write.sum (bytes), or None"""
    import csv
    try:
        per = {}
        with open(path) as f:
            rows = [r for r in csv.reader(f) if len(r) > 14 and r[0].isdigit()]
        for r in rows:
            if r[12] in ("dram__bytes_read.sum", "dram__bytes_write.sum") and kernel in r[4]:
                per[r[0]] = per.get(r[0], 0.0) + float(r[14].replace(",", ""))
        return sum(per.values()) / len(per) if per else None
    except OSError:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--engine", default="auto", choices=["auto", "split", "fused", "lockstep"])
    ap.add_argument("--games", type=int, default=4096, help="concurrent games per GPU = games a step runs to completion")
    ap.add_argument("--e2e-games", type=int, default=16384, help="games per GPU of the end-to-end generation (4 pool-fulls)")
    ap.add_argument("--gen-games", type=int, default=1200, help="games of the example_config generation (configs[3])")
    ap.add_argument("--steady-seconds", type=float, default=3.0, help="warm steady-state sample after the timed region")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--ref-seconds", type=float, default=10.0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-ref-python", action="store_true", help="skip the unmodified-reference CPU sample (about 40 s)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip generation_1200 / steady_state / engine A-B")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the timed steps to DIR/<name>.npy (see above)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs needs --impl ours")
        run_reference(args, rank)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    from connect4_b200.dist import generate_sharded, shard_games
    from connect4_b200.mcts import MCTSConfig
    from connect4_b200.neural.config import ModelConfig, NetConfig
    from connect4_b200.neural.game_pool import SelfPlayPool
    from connect4_b200.neural.model import ModelWrapper

    if args.engine != "auto":
        os.environ["C4_ENGINE"] = args.engine
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_sum_max(sums, maxs):
        a = torch.tensor(sums, dtype=torch.float64, device="cuda")
        b = torch.tensor(maxs, dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(a)
            dist.all_reduce(b, op=dist.ReduceOp.MAX)
        return [float(x) for x in a.tolist()], [float(x) for x in b.tolist()]

    z = np.load(STATE)
    model = ModelWrapper(state_dict={k: z[k] for k in z.files})
    cfg = MCTSConfig(SIMS, 19652, 1.25, 0.3, 0.25, 6)
    pool = SelfPlayPool(model, cfg, concurrent_games=args.games, seed=1000 + rank)

    def step():
        # one generation from a cold memo: fresh pool, every game from the empty board, until `games` games are done
        return pool.stream(stop_games=args.games, reset=True, cold_memo=True)

    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    tot = dict(positions=0, evals=0, device_ms=0.0, games=0, memo_hits=0, launches=0, passes=0)
    tree_ms_sum = net_ms_sum = 0.0
    t_wall = time.perf_counter()
    for _ in range(args.steps):
        r = step()
        for k in tot:
            tot[k] += r[k]
        engine, memo_log2 = r["engine"], r["memo_log2"]
        tree_ms_sum += r["tree_ms"]
        net_ms_sum += r["net_ms"]
    barrier()
    t_wall = time.perf_counter() - t_wall
    clocks = sampler.stop() if sampler else None
    (positions, evals, games, hits), (dev_ms,) = reduce_sum_max(
        [tot["positions"], tot["evals"], tot["games"], tot["memo_hits"]], [tot["device_ms"]])
    secs = dev_ms / 1000.0
    value = positions / secs

    # end to end through the public API with host buffers: one whole generation, records back on the host
    e2e = e2e_rec = None
    if not args.no_e2e:
        n_e2e = args.e2e_games * world
        start = (torch.zeros(args.e2e_games, dtype=torch.int64).pin_memory(),               # host-resident (pinned) inputs:
                 torch.zeros(args.e2e_games, dtype=torch.int64).pin_memory())               # every game from the empty board
        pool2 = SelfPlayPool(model, cfg, concurrent_games=args.games, seed=5000)
        if world == 1:
            pool2.generate_records(min(64, args.e2e_games), start=(start[0][:64], start[1][:64]))   # warm the path
        else:
            generate_sharded(pool2, 64 * world, dst=0)                       # (incl. the communicator and the sort kernels)
        first = None
        for rep in range(2):                                                 # the first run warms every kernel at full size (sort, gather, copy)
            pool2.engine.clear_memo()
            barrier()
            t0 = time.perf_counter()
            if world == 1:
                rec = pool2.generate_records(args.e2e_games, start=start)
            else:
                # every rank plays its share (global game ids, so the generation does not depend on N), then the NCCL
                # all-gather of the records and the device-side sort: every GPU ends with the whole generation in HBM and rank 0
                # (the reference collects the games in one process, neural/training.py:112-133) with the whole generation on its host
                phases = {}
                rec = generate_sharded(pool2, n_e2e, dst=0, timing=phases)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            (n_rec,), (dt_max,) = reduce_sum_max([len(rec) if rec is not None else 0], [dt])
            if first is None:
                first = dt_max
                del rec
        n_rec = int(n_rec)                                                   # N > 1: rank 0 holds the whole job's records
        e2e = {"value": n_rec / dt_max, "unit": UNIT,
               "h2d_bytes_per_step": int(2 * 8 * args.e2e_games) if world == 1 else 0,
               "d2h_bytes_per_step": int(n_rec * 64),
               "what": ("SelfPlayPool.generate_records(%d games on %d slots, pinned host start positions) -> host records; "
                        "cold memo; wall clock of the whole generation incl. the drain of the last games; second of two such generations" % (
                            args.e2e_games, args.games)) if world == 1 else
                       ("dist.generate_sharded(%d games = %d per GPU on %d slots): generation + NCCL all-gather of all "
                        "records to every GPU + device-side sort + copy of the whole generation to rank 0's host; cold memo; wall "
                        "clock, max over ranks; second of two such generations" % (n_e2e, args.e2e_games, args.games)),
               "records": n_rec, "seconds": dt_max, "seconds_first_run": first,
               "rank0_phase_seconds": {k: round(v, 4) for k, v in phases.items()} if world > 1 else None,
               "records_sha256_16": digest_records(rec) if world > 1 and rec is not None else None}
        pool2.engine.close()
        e2e_rec = rec if args.dump_outputs else None
        del rec
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, r, e2e_rec)

    extras = {}
    if not args.no_extras:
        # BASELINE configs[3]: the reference's example_config generation (oinkoink/data/example_config.py:8-16) sharded over N
        torch.manual_seed(0)                                                 # the same random-init network on every rank
        model64 = ModelWrapper(ModelConfig(net_config=NetConfig(filters=64, n_fc_layers=6, n_residuals=6)))
        n_local = shard_games(args.gen_games, rank, world)[0]
        pool3 = SelfPlayPool(model64, cfg, concurrent_games=max(1, n_local), seed=0)
        best = None
        for rep in range(2):                                                 # the first run also warms the path
            pool3.engine.clear_memo()
            barrier()
            t0 = time.perf_counter()
            rec = generate_sharded(pool3, args.gen_games, dst=0)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            (_,), (dt_max,) = reduce_sum_max([0.0], [dt])
            best = dt_max
        if rank == 0:
            extras["generation_1200"] = {
                "games": args.gen_games, "n_gpus": world, "net": "example_config 64f/6r/6fc (random init, torch.manual_seed(0))",
                "seconds": best, "positions": int(len(rec)), "positions_per_sec": len(rec) / best,
                "records_sha256_16": digest_records(rec), "scaling": "strong",
                "what": "dist.generate_sharded(dst=0): games g -> rank g % N, NCCL all-gather of the records, device-side sort, "
                        "copy of the generation to rank 0's host"}
        pool3.engine.close()
        # warm regime, context only: continue one pool for a few seconds so the memo holds millions of positions
        step()
        t_warm = 0.0
        while t_warm < args.steady_seconds * 1e3:
            r = pool.stream(max_ms=500.0)
            t_warm += r["device_ms"]
        (wp,), (wms,) = reduce_sum_max([r["positions"]], [r["device_ms"]])
        extras["steady_state"] = {"value": wp / wms * 1e3, "unit": UNIT,
                                  "memo_hit_rate": r["memo_hits"] / max(1, r["memo_hits"] + r["evals"]),
                                  "after_device_seconds_of_play": t_warm / 1e3,
                                  "note": "memo warmed by seconds of play with one network: not reachable in a real generation"}
        if world == 1 and args.engine == "auto":
            ab = []
            for other in ("split", "fused", "lockstep"):
                if other == engine:
                    continue
                os.environ["C4_ENGINE"] = other
                p4 = SelfPlayPool(model, cfg, concurrent_games=args.games, seed=1000)
                rr = [p4.stream(stop_games=args.games, reset=True, cold_memo=True) for _ in range(3)][1:]
                if rr[0]["engine"] == other:
                    ab.append({"engine": other, "value": sum(x["positions"] for x in rr) / sum(x["device_ms"] for x in rr) * 1e3,
                               "unit": UNIT, "memo_hit_rate": sum(x["memo_hits"] for x in rr) / max(1, sum(x["memo_hits"] + x["evals"] for x in rr))})
                p4.engine.close()
            os.environ.pop("C4_ENGINE")
            extras["engine_ab"] = {"what": "the same cold generation on this package's other engines", "runs": ab}

    if rank == 0:
        peak_tf, peak_hbm, peak_src = peaks()
        flops = model.flops_per_position
        step_ms = 1000.0 * secs / args.steps
        # kernels of the engine per step: the split engine cuts a step into time slices (adaptive tower count), one launch each;
        # every c4_selfplay_stream call reports its launches (2 of them are the k_sum_stats bookkeeping kernels)
        eng_launches = max(args.steps, int(tot["launches"]) - 2 * args.steps) if engine == "split" else args.steps
        n_launch = eng_launches * world
        launch_ms = 1000.0 * secs / eng_launches
        tf = evals * flops / secs / 1e12 / world                              # per GPU
        tree_bytes = positions * SIMS * 1280.0 + (evals + hits) * 64.0
        gbs = tree_bytes / secs / 1e9 / world
        if engine in ("fused", "split"):
            # persistent engines: the kernel(s) run for the whole step, so launch duration = step time
            if engine == "fused":
                kname_t = kname_h = "k_fused<OpFP16,selfplay> (persistent: tree warps + tcgen05 tower per SM, one launch per step)"
                where_t = where_h = ""
            else:
                sms = torch.cuda.get_device_properties(local).multi_processor_count
                if "C4_SP_NET_CTAS" in os.environ or os.environ.get("C4_SP_ADAPT") == "0":
                    n_net = int(os.environ.get("C4_SP_NET_CTAS", (sms * 72 + 74) // 148))
                    n_t, n_h = "%d" % n_net, "%d" % (sms - n_net)
                else:                                                 # adaptive: chosen per 25 ms slice from the previous slice's load
                    n_t = "%d..%d (adaptive, per slice)" % ((sms * 40 + 74) // 148, (sms * 96 + 74) // 148)
                    n_h = "%d..%d (adaptive, per slice)" % (sms - (sms * 96 + 74) // 148, sms - (sms * 40 + 74) // 148)
                kname_h = "k_sp_one<OpFP16,32,selfplay>, tree CTAs (%s of %d SMs: 31 game warps + 1 mail warp each)" % (n_h, sms)
                kname_t = "k_sp_one<OpFP16,32,selfplay>, tower CTAs (%s of %d SMs: tcgen05/TMEM tower, one leaf ring each)" % (n_t, sms)
                where_h = "; runs on %s of %d SMs, %.1f launches (time slices) per step back to back, peak = whole device" % (n_h, sms, eng_launches / args.steps)
                where_t = "; runs on %s of %d SMs, %.1f launches (time slices) per step back to back, peak = whole device" % (n_t, sms, eng_launches / args.steps)
            roof_t = {"kernel": kname_t, "bound": "tensor", "achieved": tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": tf / peak_tf,
                      "traffic": None, "peak_source": peak_src, "flops_per_eval": flops, "evals_per_launch": evals / n_launch,
                      "ms_per_launch": launch_ms, "share_of_step": 1.0,
                      "note": "network FLOPs of the step / step time; the towers run short strips (latency over fill), bound by the "
                              "per-tile issue / epilogue chain, not by the tensor pipe" + where_t}
            roof_h = {"kernel": kname_h, "bound": "hbm", "achieved": gbs, "peak": peak_hbm, "unit": "GB/s", "frac": gbs / peak_hbm,
                      "traffic": None, "peak_source": peak_src.replace("sustained bf16", "copy bandwidth"),
                      "algorithmic_bytes_per_launch": tree_bytes / n_launch, "sims_per_launch": positions * SIMS / n_launch,
                      "ms_per_launch": launch_ms, "share_of_step": 1.0,
                      "note": "1.28 KB per simulation (SURVEY.md 8d) + 64 B per memo probe; dependent-load latency bound" + where_h}
            if engine == "split" and args.games == 4096 and "C4_SP_NET_CTAS" not in os.environ:
                # DRAM bytes of this very launch shape from the ncu capture of the same command (profiles/r02_split_adapt_launches.csv:
                # `ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum -k regex:k_sp_one python bench.py --steps 1 --warmup 1
                # --no-e2e --no-cpu --no-extras`); whole kernel = both roles; no counter is read inside this run
                t = ncu_traffic(os.path.join(ROOT, "profiles", "r02_split_adapt_launches.csv"))
                if t:
                    roof_h["traffic"] = t
                    roof_h["traffic_source"] = ("profiles/r02_split_adapt_launches.csv: dram__bytes_read.sum + dram__bytes_write.sum per k_sp_one "
                                                "launch (whole kernel, both roles), ncu capture of the same workload, not this run")
            if engine == "split":
                roof_t, roof_h = roof_h, roof_t                       # `roofline` = the tree kernel: it bounds the step (tower CTAs have slack)
        else:
            # lock-step engine: per-launch figures of rank 0 from the launches sampled with CUDA events inside the timed steps
            passes = max(1, tot["passes"])
            dev_ms_rank0 = max(1e-9, tot["device_ms"])
            raw_tree, raw_net = tree_ms_sum / args.steps, net_ms_sum / args.steps
            # The sampled pass sits inside a captured launch graph; the external event records around its two kernels add a
            # few microseconds each, so the raw pairs sum to more than the device time per pass.  The event times give the
            # SPLIT between the two kernels, the step's own CUDA-event time / number of passes gives the scale.
            per_pass = dev_ms_rank0 / passes
            scale = min(1.0, per_pass / max(1e-9, raw_tree + raw_net))
            tree_ms, net_ms = raw_tree * scale, raw_net * scale
            sims_l = tot["positions"] * SIMS / passes
            bytes_l = sims_l * 1280.0 + (tot["evals"] + tot["memo_hits"]) / passes * 64.0
            evals_l = tot["evals"] / passes
            t_gbs = bytes_l / (tree_ms * 1e-3) / 1e9 if tree_ms > 0 else 0.0
            n_tf = evals_l * flops / (net_ms * 1e-3) / 1e12 if net_ms > 0 else 0.0
            roof_h = {"kernel": "k_advance<NET,selfplay> (warp-per-game tree pass)", "bound": "hbm", "achieved": t_gbs,
                      "peak": peak_hbm, "unit": "GB/s", "frac": t_gbs / peak_hbm, "traffic": None,
                      "peak_source": peak_src.replace("sustained bf16", "copy bandwidth"),
                      "algorithmic_bytes_per_launch": bytes_l, "sims_per_launch": sims_l, "ms_per_launch": tree_ms,
                      "ms_per_launch_raw_events": raw_tree, "share_of_step": tree_ms * passes / dev_ms_rank0,
                      "note": "1.28 KB per simulation (SURVEY.md 8d) + 64 B per memo probe; dependent-load latency bound, not "
                              "bandwidth bound"}
            roof_t = {"kernel": "k_net_tc<OpFP16,32> (tcgen05/TMEM)", "bound": "tensor", "achieved": n_tf, "peak": peak_tf,
                      "unit": "TFLOP/s", "frac": n_tf / peak_tf, "traffic": None, "peak_source": peak_src,
                      "flops_per_eval": flops, "evals_per_launch": evals_l, "ms_per_launch": net_ms,
                      "ms_per_launch_raw_events": raw_net, "share_of_step": net_ms * passes / dev_ms_rank0,
                      "note": "launch durations: CUDA events around the two kernels of one pass in every 8th chunk of 64 passes "
                              "(inside the captured launch graph), scaled so that tree + network = device time per pass"}
            if roof_h["share_of_step"] >= roof_t["share_of_step"]:
                roof_t, roof_h = roof_h, roof_t                       # `roofline` = the kernel with the larger share
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": step_ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "fp16", "data": "synthetic",
            "config": {"workload": WORKLOAD, "games_per_gpu": args.games, "simulations": SIMS, "memo": "cold (emptied before every step)",
                       "step": "fresh pool, finished games re-seeded at once, until %d games have completed" % args.games,
                       "engine": engine, "evaluation_memo_log2_entries": memo_log2,
                       "l2": "node pool (%.0f MB/GPU) + evaluation memo (%.1f GB) exceed L2; every step starts cold" %
                             (args.games * (SIMS + 2) * 256 / 1e6, (64 << memo_log2) / 1e9 if memo_log2 else 0.0)},
            "clocks": clocks,
            "e2e": e2e,
            "gpu_launches": int(tot["launches"] + args.steps),                  # + k_selfplay_init of every step (rank 0's count)
            "roofline": roof_t, "roofline_other": roof_h,
            "sims_per_sec": value * SIMS, "network_evals_per_sec": evals / secs,
            "memo_hit_rate": hits / max(1.0, hits + evals),
            "games_finished": games, "wall_s_timed_region": t_wall,
        }
        line.update(extras)
        if world == 1 and not args.no_cpu:
            r, cores = cpu_port(args.cpu_seconds)
            line["cpu_baseline"] = {
                "value": r["positions_per_sec"], "unit": UNIT, "cores": cores, "kind": "port",
                "sample": "%d single-threaded workers x 32 games in flight, %.0f s of self-play at 800 sims/move "
                          "(C oracle tree + torch fp32 net + per-process evaluation memo like the reference's "
                          "Evaluator.position_table); the unmodified Python reference measured 13 positions/s on 8 cores "
                          "(BASELINE.md)" % (cores, args.cpu_seconds),
                "evals_per_sec": r["evals_per_sec"]}
            if not args.no_ref_python:
                line["cpu_baseline_reference"] = reference_python()
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
