"""Exact endgame play measurements (BatchedSelfPlay(exact_endgame=max_free), DESIGN.md §14), one JSON line per figure,
beside adjudication (tools/adjudication_bench.py, DESIGN.md §12):

  games_3x3   play_games_async, 3x3, 32768 games, SimpleNN bf16, 800 simulations, eval cache emptied per batch: off,
              adjudicate 12 / 16 and exact_endgame 12 / 16, alternated.  games/h, simulations per game, checks
              (finish-graph replays) per batch, sample rows and exact rows; z_agreement of the batch graded by the 3x3
              table, and with exact play the optimal_move_rate of its exact rows graded by EndgameSolver(max_free).
  games_5x5   the same on 5x5, 16384 games, ResNetZero-20 bf16, 200 simulations: off, adjudicate 12 and exact_endgame 12,
              the net wrapped in EndgameEvaluator(net, EndgameSolver(engine, 12)) where a mode is on.
  latency     one k_selfplay_exact_endgame launch over 32768 trees of which 0, 1, 64 or 1024 qualify, with roots at
              f = max_free (10, 12, 14, 16) played out to the end; the other trees are mid-search (moves = -1).  CUDA
              events around each launch.

  python tools/exact_endgame_bench.py [--only games_3x3,games_5x5,latency] [--rounds 2] [--out FILE]
"""
import argparse
import ctypes
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from adjudication_bench import emit, gpu_info, mask_states, sp_params, summary  # noqa: E402
from dotsboxesaz_b200 import endgame, engine, samples, self_play, solver  # noqa: E402
from dotsboxesaz_b200._capi import SelfplayBuffers  # noqa: E402
from dotsboxesaz_b200.utils.utils import DotDict  # noqa: E402


def play_rounds(args, eng, settings, sims, grade=None):
    """settings: {label: (evaluator, adjudicate or None, exact_endgame or None)}; one warm-up batch each, then args.rounds
    alternating rounds"""
    n = eng.n_games
    params = sp_params(sims)
    res = {k: [] for k in settings}
    for rnd in range(args.rounds + 1):
        for label, (ev, adj, ex) in settings.items():
            bsp = self_play.BatchedSelfPlay(eng, ev, params, graph_waves=16, adaptive=True, adjudicate=adj, exact_endgame=ex)
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
                   "adjudicated": info["adjudicated"], "exact_games": info["exact_games"], "exact_rows": info["exact_rows"],
                   "sample_rows": len(batch), "errors": info["errors"]}
            if grade is not None:
                rec["z_agreement"] = solver.grade_samples(grade, batch)["z_agreement"]
            if ex is not None:
                gr = solver.grade_samples(endgame.EndgameSolver(eng, ex), batch)
                rec["exact_rows_graded"] = gr["n_solved"]
                rec["exact_optimal_move_rate"] = gr.get("optimal_move_rate")
            res[label].append(rec)
    return res


def bench_3x3(args):
    from dotsboxesaz_b200.dots_boxes.dots_boxes_nn import SimpleNN
    from dotsboxesaz_b200.nn import FusedSimpleNN
    n, nodes, sims = 32768, 4096, 800
    eng = engine.Engine((3, 3), n_games=n, max_nodes=nodes, eval_cache=self_play.eval_cache_log2_for(32, n, nodes))
    eng.set_mode(False, 4)
    torch.manual_seed(0)
    ev = FusedSimpleNN(SimpleNN(board=(3, 3)), eng, dtype=torch.bfloat16)
    table = solver.Solver(eng).solve()
    settings = {"off": (ev, None, None)}
    for m in (12, 16):
        settings["adjudicate_%d" % m] = (ev, m, None)
        settings["exact_endgame_%d" % m] = (ev, None, m)
    res = play_rounds(args, eng, settings, sims, grade=table)
    emit(args.out, {"figure": "games_3x3", "games": n, "sims": sims, "net": "SimpleNN bf16", "max_nodes": nodes,
                    "eval_cache_log2": eng.eval_cache_log2, "results": summary(res)})
    del table
    eng.close()
    torch.cuda.empty_cache()


def bench_5x5(args):
    from dotsboxesaz_b200.nn import FusedResNetZero, ResNetZero, resnet_zero_parameters
    n, nodes, sims, m = 16384, 4096, 200, 12
    eng = engine.Engine((5, 5), n_games=n, max_nodes=nodes, eval_cache=self_play.eval_cache_log2_for(72, n, nodes))
    eng.set_mode(False, 4)
    torch.manual_seed(0)
    net = FusedResNetZero(ResNetZero(DotDict({"nn": {"model_parameters": resnet_zero_parameters((5, 5))}})), eng, dtype=torch.bfloat16)
    wrapped = endgame.EndgameEvaluator(net, endgame.EndgameSolver(eng, m))
    settings = {"off": (net, None, None), "adjudicate_%d" % m: (wrapped, m, None), "exact_endgame_%d" % m: (wrapped, None, m)}
    res = play_rounds(args, eng, settings, sims)
    emit(args.out, {"figure": "games_5x5", "games": n, "sims": sims, "net": "ResNetZero-20 bf16", "max_nodes": nodes,
                    "eval_cache_log2": eng.eval_cache_log2, "results": summary(res)})
    eng.close()
    torch.cuda.empty_cache()


def bench_latency(args):
    n = 32768
    for board in ((3, 3), (5, 5)):
        eng = engine.Engine(board, n_games=n, max_nodes=16)
        dev, A = eng.device, eng.A
        n_moves = 17  # a playout from f <= 16 writes at most 16 rows from move index 0
        ptr = lambda t: ctypes.c_void_p(t.data_ptr())
        t = dict(inv_temp=torch.ones((n_moves,), dtype=torch.float64, device=dev),
                 uniforms=torch.rand((n_moves, n), dtype=torch.float64, device=dev),
                 reads_by_k=torch.ones((A + 1,), dtype=torch.int32, device=dev),
                 searching=torch.ones((n,), dtype=torch.int8, device=dev),
                 move_idx=torch.zeros((n,), dtype=torch.int64, device=dev),
                 moves=torch.full((n,), -1, dtype=torch.int32, device=dev),
                 h_states=torch.zeros((n_moves, n, 4), dtype=torch.int64, device=dev),
                 h_visits=torch.zeros((n_moves, n, A), dtype=torch.int32, device=dev),
                 h_active=torch.zeros((n_moves, n), dtype=torch.int8, device=dev),
                 h_moves=torch.zeros((n_moves, n), dtype=torch.int32, device=dev),
                 h_stats=torch.zeros((n_moves, n, 8), dtype=torch.int32, device=dev),
                 h_q=torch.zeros((n_moves, n), dtype=torch.float32, device=dev),
                 noise_buf=torch.zeros((n, A), dtype=torch.float64, device=dev),
                 reads=torch.zeros((n,), dtype=torch.int32, device=dev),
                 left=torch.zeros((1,), dtype=torch.int32, device=dev))
        bufs = SelfplayBuffers(n_moves=n_moves, noise=None, **{k: ptr(v) for k, v in t.items()})
        margin = torch.full((n,), -128, dtype=torch.int8, device=dev)
        for mf in (10, 12, 14, 16):
            eg = endgame.EndgameSolver(eng, mf)
            for k in (0, 1, 64, 1024):
                roots = eng.new_states(n)
                if k:
                    roots[:k] = mask_states(eng, mf, k, seed=mf * 1000 + k)
                eng.reset_roots(roots.contiguous())
                t["moves"].fill_(-1)
                t["moves"][:k] = 0
                times = []
                for r in range(args.reps + 3):
                    t["searching"].fill_(1)
                    t["move_idx"].zero_()
                    margin.fill_(-128)
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    eg.play_out(bufs, margin)
                    b.record()
                    b.synchronize()
                    if r >= 3:
                        times.append(a.elapsed_time(b) * 1e3)
                assert int((margin[:k] != -128).sum()) == k and int((margin[k:] != -128).sum()) == 0
                rows = int(t["move_idx"][:k].sum()) + k  # rows written by the last launch
                emit(args.out, {"figure": "latency", "board": "%dx%d" % board, "trees": n, "max_free": mf, "free_edges": mf,
                                "qualifying": k, "rows_written": rows, "median_us": float(np.median(times)),
                                "min_us": float(np.min(times))})
        eng.close()


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--rounds", type=int, default=2, help="alternating timed batches per setting (after one warm-up each)")
    ap.add_argument("--reps", type=int, default=50, help="timed launches per latency figure")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    ap.add_argument("--only", default="games_3x3,games_5x5,latency")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("exact_endgame_bench.py measures self-play on the GPU: no CUDA device")
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
