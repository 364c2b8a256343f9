"""Adjudication measurements (BatchedSelfPlay(adjudicate=max_free), DESIGN.md §12), one JSON line per figure:

  games_3x3   play_games_async, 3x3, 32768 games, SimpleNN bf16, 800 simulations, eval cache emptied per batch:
              adjudication off and at max_free 8, 10, 12, 16, alternated.  games/h, simulations per game, checks
              (finish-graph replays) per batch, sample rows, and z_agreement of the batch graded by the 3x3 table.
  games_5x5   the same on 5x5, 16384 games, ResNetZero-20 bf16, 200 simulations: off, and at max_free 8, 10, 12 with the
              net wrapped in EndgameEvaluator(net, EndgameSolver(engine, max_free)).
  latency     one k_selfplay_adjudicate launch over 32768 trees of which 1, 64 or 1024 qualify, with roots at
              f = max_free (10, 12, 14, 16); the other trees are mid-search (moves = -1).  CUDA events around each launch.

  python tools/adjudication_bench.py [--only games_3x3,games_5x5,latency] [--rounds 2] [--out FILE]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from dotsboxesaz_b200 import endgame, engine, samples, self_play, solver  # noqa: E402
from dotsboxesaz_b200._capi import SelfplayBuffers  # noqa: E402
from dotsboxesaz_b200.utils.utils import DotDict  # noqa: E402


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as exc:  # noqa: BLE001
        q = "unknown (%s)" % exc
    return q


def emit(out, rec):
    line = json.dumps(rec)
    print(line, flush=True)
    if out:
        with open(out, "a") as f:
            f.write(line + "\n")


def sp_params(sims):
    return DotDict({"self_play": {"reuse_mcts_tree": True, "noise": (0.8, 0.25),
                                  "mcts": {"mcts_num_read": sims, "mcts_cpuct": (1.25, 19652), "temperature": {0: 1.0, 12: 0.02},
                                           "max_async_searches": 1}}})


def play_rounds(args, eng, evaluators, sims, grade=None):
    """evaluators: {label: (evaluator, max_free or None)}; one warm-up batch each, then args.rounds alternating rounds"""
    n = eng.n_games
    params = sp_params(sims)
    res = {k: [] for k in evaluators}
    for rnd in range(args.rounds + 1):
        for label, (ev, mf) in evaluators.items():
            bsp = self_play.BatchedSelfPlay(eng, ev, params, graph_waves=16, adaptive=True, adjudicate=mf)
            eng.clear_eval_cache()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            info = bsp.play_games_async(range(n), seed=rnd)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            if rnd == 0:
                continue  # warm-up: graph captures for this evaluator
            batch = samples.batch_from_selfplay(bsp, 0)
            rec = {"games_per_hour": n / dt * 3600.0, "seconds": dt, "sims_per_game": info["sims"] / n, "checks": info["checks"],
                   "adjudicated": info["adjudicated"], "sample_rows": len(batch), "errors": info["errors"]}
            if grade is not None:
                rec["z_agreement"] = solver.grade_samples(grade, batch)["z_agreement"]
            res[label].append(rec)
    return res


def summary(res):
    return {k: {"median_games_per_hour": float(np.median([r["games_per_hour"] for r in v])), "runs": v} for k, v in res.items()}


def bench_3x3(args):
    from dotsboxesaz_b200.dots_boxes.dots_boxes_nn import SimpleNN
    from dotsboxesaz_b200.nn import FusedSimpleNN
    n, nodes, sims = 32768, 4096, 800
    eng = engine.Engine((3, 3), n_games=n, max_nodes=nodes, eval_cache=self_play.eval_cache_log2_for(32, n, nodes))
    eng.set_mode(False, 4)
    torch.manual_seed(0)
    ev = FusedSimpleNN(SimpleNN(board=(3, 3)), eng, dtype=torch.bfloat16)
    table = solver.Solver(eng).solve()
    evs = {"off": (ev, None)}
    evs.update({"max_free_%d" % m: (ev, m) for m in (8, 10, 12, 16)})
    res = play_rounds(args, eng, evs, sims, grade=table)
    emit(args.out, {"figure": "games_3x3", "games": n, "sims": sims, "net": "SimpleNN bf16", "max_nodes": nodes,
                    "eval_cache_log2": eng.eval_cache_log2, "results": summary(res)})
    del table
    eng.close()
    torch.cuda.empty_cache()


def bench_5x5(args):
    from dotsboxesaz_b200.nn import FusedResNetZero, ResNetZero, resnet_zero_parameters
    n, nodes, sims = 16384, 4096, 200
    eng = engine.Engine((5, 5), n_games=n, max_nodes=nodes, eval_cache=self_play.eval_cache_log2_for(72, n, nodes))
    eng.set_mode(False, 4)
    torch.manual_seed(0)
    net = FusedResNetZero(ResNetZero(DotDict({"nn": {"model_parameters": resnet_zero_parameters((5, 5))}})), eng, dtype=torch.bfloat16)
    evs = {"off": (net, None)}
    evs.update({"max_free_%d" % m: (endgame.EndgameEvaluator(net, endgame.EndgameSolver(eng, m)), m) for m in (8, 10, 12)})
    res = play_rounds(args, eng, evs, sims)
    emit(args.out, {"figure": "games_5x5", "games": n, "sims": sims, "net": "ResNetZero-20 bf16", "max_nodes": nodes,
                    "eval_cache_log2": eng.eval_cache_log2, "results": summary(res)})
    eng.close()
    torch.cuda.empty_cache()


def mask_states(eng, n_free, n, seed):
    """n states with exactly n_free free real edges chosen at random"""
    dev = eng.device
    gen = torch.Generator(device=dev)
    gen.manual_seed(seed)
    cols, plane = eng.C + 1, (eng.L + 1) * (eng.C + 1)
    real = torch.tensor([a for a in range(2 * plane) if (a < plane and a % cols < eng.C) or (a >= plane and (a - plane) // cols < eng.L)],
                        dtype=torch.int64, device=dev)
    ranks = torch.rand((n, real.numel()), generator=gen, device=dev).argsort(1)
    bits = torch.zeros((n, 128), dtype=torch.int64, device=dev)
    bits[:, real] = (ranks >= n_free).long()
    sh = torch.arange(64, device=dev)
    st = eng.new_states(1).repeat(n, 1)
    st[:, 0] = (bits[:, :64] << sh).sum(1)
    st[:, 1] = (bits[:, 64:] << sh).sum(1)
    return st.contiguous()


def bench_latency(args):
    n = 32768
    for board in ((3, 3), (5, 5)):
        eng = engine.Engine(board, n_games=n, max_nodes=16)
        dev, A = eng.device, eng.A
        ptr = lambda t: ctypes.c_void_p(t.data_ptr())
        searching = torch.ones((n,), dtype=torch.int8, device=dev)
        moves = torch.full((n,), -1, dtype=torch.int32, device=dev)
        reads = torch.zeros((n,), dtype=torch.int32, device=dev)
        left = torch.zeros((1,), dtype=torch.int32, device=dev)
        margin = torch.full((n,), -128, dtype=torch.int8, device=dev)
        dummy = torch.zeros((n, A), dtype=torch.float64, device=dev)
        d = ptr(dummy)
        bufs = SelfplayBuffers(n_moves=1, inv_temp=d, uniforms=d, noise=None, reads_by_k=d, searching=ptr(searching), move_idx=d,
                               moves=ptr(moves), h_states=d, h_visits=d, h_active=d, h_moves=d, h_stats=d, h_q=d, noise_buf=d,
                               reads=ptr(reads), left=ptr(left))
        for mf in (10, 12, 14, 16):
            eg = endgame.EndgameSolver(eng, mf)
            for k in (0, 1, 64, 1024):
                roots = eng.new_states(n)
                if k:
                    roots[:k] = mask_states(eng, mf, k, seed=mf * 1000 + k)
                eng.reset_roots(roots.contiguous())
                moves.fill_(-1)
                moves[:k] = 0
                times = []
                for r in range(args.reps + 3):
                    searching.fill_(1)
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    eg.adjudicate(bufs, margin)
                    b.record()
                    b.synchronize()
                    if r >= 3:
                        times.append(a.elapsed_time(b) * 1e3)
                assert int((margin[:k] != -128).sum()) == k
                emit(args.out, {"figure": "latency", "board": "%dx%d" % board, "trees": n, "max_free": mf, "free_edges": mf,
                                "qualifying": k, "median_us": float(np.median(times)), "min_us": float(np.min(times))})
        eng.close()


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--rounds", type=int, default=2, help="alternating timed batches per setting (after one warm-up each)")
    ap.add_argument("--reps", type=int, default=50, help="timed launches per latency figure")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    ap.add_argument("--only", default="games_3x3,games_5x5,latency")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("adjudication_bench.py measures self-play on the GPU: no CUDA device")
    emit(args.out, {"figure": "gpu", "gpu": gpu_info()})
    parts = args.only.split(",")
    if "latency" in parts:
        bench_latency(args)
    if "games_3x3" in parts:
        bench_3x3(args)
    if "games_5x5" in parts:
        bench_5x5(args)


if __name__ == "__main__":
    main()
