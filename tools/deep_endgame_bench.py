"""Deep-tier endgame measurements (DeepEndgameSolver, dbaz_endgame_deep_moves, DESIGN.md §13), one JSON line per figure.
The first line gives the card's name, power limit and max SM clock, read in the same run.

  rate      per-position time and successor reads/s (f 2^(f-1) per position) at f = 17, 20, 22, 24, 26, 28, 30, 32 on 4x4,
            5x5 and 7x7 (random masks), 8 GiB workspace: one position, and full passes (as many positions as the workspace
            holds, at most 65 535).  Host clock around DeepEndgameSolver.moves, which synchronises; one warm-up call each.
  full      the empty 3x4 board through the deep tier (f = 31, one position) against Solver.solve() on 3x4, alternated.
  parent    Solver.solve() on 3x4 with this tree's library and with the library given by --parent-lib, alternated.
  grade     a 5x5 self-play batch (play_games_async, 4096 games, 200 simulations, FakeNetEvaluator) graded with
            EndgameSolver(eng, 16) and DeepEndgameSolver with max_free 20 and 24: rows solved and seconds.

  python tools/deep_endgame_bench.py [--only rate,full,parent,grade] [--parent-lib PATH] [--out FILE]
"""
import argparse
import copy
import ctypes as C
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from dotsboxesaz_b200 import _capi, endgame, engine, solver  # noqa: E402

GIB = 1 << 30


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


def real_actions(L, C_):
    cols, plane = C_ + 1, (L + 1) * (C_ + 1)
    return [a for a in range(2 * plane) if (a < plane and a % cols < C_) or (a >= plane and (a - plane) // cols < L)]


def mask_states(eng, n_free, n, seed):
    """n states with exactly n_free free real edges chosen at random; both players' scores even"""
    dev = eng.device
    gen = torch.Generator(device=dev)
    gen.manual_seed(seed)
    real = torch.tensor(real_actions(eng.L, eng.C), dtype=torch.int64, device=dev)
    ranks = torch.rand((n, real.numel()), generator=gen, device=dev).argsort(1)
    bits = torch.zeros((n, 128), dtype=torch.int64, device=dev)
    bits[:, real] = (ranks >= n_free).long()
    sh = torch.arange(64, device=dev)
    st = eng.new_states(1).repeat(n, 1)
    st[:, 0] = (bits[:, :64] << sh).sum(1)
    st[:, 1] = (bits[:, 64:] << sh).sum(1)
    return st.contiguous()


def timed(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t


def bench_rate(out):
    ws = 8 * GIB
    for board in ((4, 4), (5, 5), (7, 7)):
        eng = engine.Engine(board, n_games=1, max_nodes=16)
        deep = endgame.DeepEndgameSolver(eng, 32, workspace_bytes=ws)
        for f in (17, 20, 22, 24, 26, 28, 30, 32):
            full = min(ws // ((1 << f) + _capi.ENDGAME_DEEP_GEOM_BYTES), 65535)
            for n in (1, full):
                st = mask_states(eng, f, n, seed=f * 100 + n)
                deep.moves(st)  # warm-up
                sec = timed(lambda: deep.moves(st))
                reads = n * f * (1 << (f - 1))
                emit(out, {"figure": "rate", "board": "%dx%d" % board, "f": f, "positions": n, "seconds": sec,
                           "us_per_position": 1e6 * sec / n, "reads_per_s": reads / sec})
        del deep
        eng.close()
        torch.cuda.empty_cache()


def bench_full(out, reps=5):
    eng = engine.Engine((3, 4), n_games=1, max_nodes=16)
    s = solver.Solver(eng)
    table = torch.empty((1 << 31,), dtype=torch.int8, device=eng.device)
    deep = endgame.DeepEndgameSolver(eng, 31, workspace_bytes=(1 << 31) + _capi.ENDGAME_DEEP_GEOM_BYTES)
    root = eng.new_states(1)
    s.solve(table)
    deep.moves(root)
    t_solve, t_deep = [], []
    for _ in range(reps):
        t_solve.append(timed(lambda: s.solve(table)) * 1e3)
        t_deep.append(timed(lambda: deep.moves(root)) * 1e3)
    same = torch.equal(deep.moves(root)[0], s.moves(root)[0])
    emit(out, {"figure": "full", "board": "3x4", "solver_solve_ms": sorted(t_solve), "deep_f31_ms": sorted(t_deep),
               "median_ratio": sorted(t_deep)[reps // 2] / sorted(t_solve)[reps // 2], "identical_moves": same})
    del table, deep, s
    eng.close()
    torch.cuda.empty_cache()


def load_lib(path):
    lib = C.CDLL(os.path.abspath(path))
    for name, (res, args) in _capi.SYMBOLS.items():
        fn = getattr(lib, name, None)
        if fn is not None:
            fn.restype = res
            fn.argtypes = args
    return lib


def bench_parent(out, path, reps=7):
    libs = {"change": _capi.load(), "parent": load_lib(path)}
    engs = {}
    for k, lib in libs.items():
        saved = _capi._lib
        _capi._lib = lib
        try:
            engs[k] = engine.Engine((3, 4), n_games=1, max_nodes=16)
        finally:
            _capi._lib = saved
    table = torch.empty((1 << 31,), dtype=torch.int8, device=engs["change"].device)
    times = {k: [] for k in engs}
    tables = {}
    for k, e in engs.items():
        solver.Solver(e).solve(table)
        tables[k] = table[::4099].clone()
    for _ in range(reps):
        for k, e in engs.items():
            s = solver.Solver(e)
            times[k].append(timed(lambda: s.solve(table)) * 1e3)
    emit(out, {"figure": "parent", "board": "3x4", "solve_ms": {k: sorted(v) for k, v in times.items()},
               "median_ms": {k: sorted(v)[reps // 2] for k, v in times.items()},
               "sampled_tables_equal": torch.equal(tables["change"], tables["parent"])})
    for e in engs.values():
        e.close()
    del table
    torch.cuda.empty_cache()


def bench_grade(out, n=4096, sims=200):
    from dotsboxesaz_b200 import configuration, samples, self_play
    p = copy.deepcopy(configuration.simple)
    p.self_play.mcts.mcts_num_read = sims
    eng = engine.Engine((5, 5), n_games=n, max_nodes=4 * sims + 64, eval_cache=20)
    bsp = self_play.BatchedSelfPlay(eng, engine.FakeNetEvaluator(0), p, graph_waves=4, pending=1, adaptive=True)
    bsp.play_games_async(list(range(n)), seed=1)
    batch = samples.batch_from_selfplay(bsp, 0)
    for mf in (16, 20, 24):
        es = endgame.EndgameSolver(eng, 16) if mf == 16 else endgame.DeepEndgameSolver(eng, mf)
        solver.grade_samples(es, batch)  # warm-up (allocates the workspace)
        res = {}
        sec = timed(lambda: res.update(solver.grade_samples(es, batch)))
        emit(out, {"figure": "grade", "board": "5x5", "games": n, "sims": sims, "max_free": mf, "rows": res["n"],
                   "rows_solved": res["n_solved"], "seconds": sec, "optimal_move_rate": res["optimal_move_rate"],
                   "z_agreement": res["z_agreement"]})
        del es
        torch.cuda.empty_cache()
    eng.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default="rate,full,parent,grade")
    ap.add_argument("--parent-lib", default=None)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("deep_endgame_bench needs a CUDA device")
    emit(a.out, {"figure": "gpu", "name_power_limit_max_sm_clock": gpu_info()})
    only = a.only.split(",")
    if "full" in only:
        bench_full(a.out)
    if "parent" in only and a.parent_lib:
        bench_parent(a.out, a.parent_lib)
    if "rate" in only:
        bench_rate(a.out)
    if "grade" in only:
        bench_grade(a.out)


if __name__ == "__main__":
    main()
