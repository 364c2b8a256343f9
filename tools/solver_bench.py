"""Exact-solver measurements (dotsboxesaz_b200/solver.py, DESIGN.md §10), one JSON line per figure:

  solve        time of Solver.solve() (fill, one k_solver_layer per popcount layer, sentinel check) for every supported
               board, with the root's final margin and outcome
  kernels      k_solver_moves / k_solver_eval throughput at 4096 and 32768 states of 3x3 and 3x4 (positions from random
               games), CUDA events around 200 launches
  search       Engine.run_search sims/s on 3x3, 4096 trees x 800 simulations from random roots 0 .. 12 plies deep, through the
               production schedule of bench.py
               (eval cache of 2^24 entries emptied per search, compact rows, adaptive ladder, device-driven loop, max_inline
               4, Dirichlet noise 0.8 / 0.25), SolverEvaluator against FakeNetEvaluator, alternated

  python tools/solver_bench.py [--skip-large] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from dotsboxesaz_b200 import engine, solver  # noqa: E402

ROOT_PLIES = 12  # search roots 0 .. 12 plies deep, as bench.py's synthetic roots
SUPPORTED = ([(1, c) for c in range(1, 11)] + [(l, 1) for l in range(2, 11)] + [(2, c) for c in range(2, 7)] +
             [(l, 2) for l in range(3, 7)] + [(3, 3), (3, 4), (4, 3)])


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


def random_states(eng, n, seed, max_plies=None):
    """positions from uniform random games stopped after 0 .. max_plies plies (default: any length)"""
    gen = torch.Generator(device=eng.device)
    gen.manual_seed(seed)
    E = eng.L * (eng.C + 1) + eng.C * (eng.L + 1)
    max_plies = E - 1 if max_plies is None else max_plies
    depth = torch.randint(0, max_plies + 1, (n,), generator=gen, device=eng.device)
    st = eng.new_states(n)
    for ply in range(max_plies):
        valid = eng.valid_moves(st).double()
        live = (depth > ply) & (eng.result(st) == 2) & (valid.sum(1) > 0)
        mv = torch.multinomial(valid + (valid.sum(1, keepdim=True) == 0).double(), 1, generator=gen).reshape(-1)
        eng.play(st, torch.where(live, mv, torch.full_like(mv, -1)).int())
    return st


def bench_solve(args):
    boards = [b for b in SUPPORTED if not (args.skip_large and b[0] * (b[1] + 1) + b[1] * (b[0] + 1) > 28)]
    for board in boards:
        eng = engine.Engine(board, n_games=1, max_nodes=16)
        s = solver.Solver(eng)
        reps = 5 if s.E <= 26 else 2
        times = []
        for _ in range(reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            s.solve(s.table)  # synchronises
            times.append(time.perf_counter() - t0)
        root = eng.new_states(1)
        m = int(s.margin(root)[0])
        emit(args.out, {"figure": "solve", "board": "%dx%d" % board, "edges": s.E, "table_bytes": 1 << s.E, "seconds_min": min(times),
                        "seconds_all": times, "successor_reads_G": s.E * 2 ** (s.E - 1) / 1e9, "root_final_margin": m,
                        "root_outcome": int(np.sign(m))})
        del s
        eng.close()
        torch.cuda.empty_cache()


def time_launches(fn, reps=200):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e3 / reps  # microseconds per launch


def bench_kernels(args):
    for board in [(3, 3)] + ([] if args.skip_large else [(3, 4)]):
        eng = engine.Engine(board, n_games=1, max_nodes=16)
        s = solver.Solver(eng).solve()
        for n in (4096, 32768):
            st = random_states(eng, n, seed=n)
            mm = torch.empty((n, eng.A), dtype=torch.int8, device=eng.device)
            mg = torch.empty((n,), dtype=torch.int8, device=eng.device)
            P = torch.empty((n, eng.A), dtype=torch.float32, device=eng.device)
            V = torch.empty((n,), dtype=torch.float32, device=eng.device)
            us_moves = time_launches(lambda: eng._ck(eng.lib.dbaz_solver_moves(eng._h, engine._ptr(s.table), engine._ptr(st), engine._ptr(mm),
                                                                               engine._ptr(mg), n, eng._stream())))
            us_eval = time_launches(lambda: s.evaluate(eng, st, P, V, 0))
            us_fake = time_launches(lambda: eng.fake_nn(st, 0, P, V))
            emit(args.out, {"figure": "kernels", "board": "%dx%d" % board, "states": n, "k_solver_moves_us": us_moves,
                            "k_solver_moves_states_per_s": n / us_moves * 1e6, "k_solver_eval_us": us_eval,
                            "k_solver_eval_states_per_s": n / us_eval * 1e6, "k_fake_nn_us": us_fake})
        del s
        eng.close()
        torch.cuda.empty_cache()


def bench_search(args):
    n, sims = 4096, 800
    eng = engine.Engine((3, 3), n_games=n, max_nodes=sims + 8, eval_cache=24)
    eng.set_mode(False, 4)
    s = solver.Solver(eng).solve()
    evs = {"solver_outcome": solver.SolverEvaluator(s, "outcome"), "solver_margin": solver.SolverEvaluator(s, "margin"),
           "fake": engine.FakeNetEvaluator(0)}
    rng = np.random.RandomState(1234)
    roots = random_states(eng, n, seed=1234, max_plies=ROOT_PLIES)  # never terminal at this depth
    valid = eng.valid_moves(roots).cpu().numpy()
    noise = torch.from_numpy(rng.dirichlet(np.ones(eng.A) * 0.8, size=n) * valid).to(eng.device)

    def run(ev):
        eng.reset_roots(roots)
        eng.clear_eval_cache()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        eng.run_search(sims, ev, noise=noise, coeff=0.25, graph_waves=8, adaptive=True)
        eng.root_visits()
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    for ev in evs.values():  # capture and warm up every ladder
        run(ev)
        run(ev)
    res = {k: [] for k in evs}
    for _ in range(args.rounds):
        for k, ev in evs.items():
            res[k].append(n * sims / run(ev))
    info = eng.status()
    emit(args.out, {"figure": "search", "board": "3x3", "trees": n, "sims": sims, "sims_per_s": {k: sorted(v) for k, v in res.items()},
                    "median_sims_per_s": {k: float(np.median(v)) for k, v in res.items()}, "device_loop": eng.device_loop,
                    "errors": info["errors"]})
    eng.close()


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--skip-large", action="store_true", help="only boards of at most 28 edges")
    ap.add_argument("--rounds", type=int, default=5, help="alternating timed searches per evaluator")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    ap.add_argument("--only", default="solve,kernels,search")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("solver_bench.py measures the GPU kernels: no CUDA device")
    emit(args.out, {"figure": "gpu", "gpu": gpu_info()})
    parts = args.only.split(",")
    if "solve" in parts:
        bench_solve(args)
    if "kernels" in parts:
        bench_kernels(args)
    if "search" in parts:
        bench_search(args)


if __name__ == "__main__":
    main()
