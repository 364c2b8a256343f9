"""Endgame-solver measurements (dotsboxesaz_b200/endgame.py, DESIGN.md §11), one JSON line per figure:

  kernels      k_endgame_eval / k_endgame_moves time against the number of free edges f (4, 8, 10, 12, 14, 16: every row
               has exactly f, random masks) and the batch (4096, 32768 rows) on 5x5 and 7x7, max_free 16; k_fake_nn on the
               same rows for scale.  CUDA events around `--reps` launches.
  search       Engine.run_search sims/s on 5x5, 16384 trees x 800 simulations, through the production schedule of
               bench.py (eval cache of 2^24 entries emptied per search, compact rows, adaptive ladder, device-driven loop,
               max_inline 4, Dirichlet noise 0.8 / 0.25): FakeNetEvaluator alone and wrapped in EndgameEvaluator with
               max_free 8 and 12, alternated.  Two root sets: 0 .. 12 plies deep (bench.py's synthetic roots) and
               36 .. 44 plies deep (16 .. 24 free edges, so the leaves reach the solvable range).

  python tools/endgame_bench.py [--only kernels,search] [--out FILE]
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

from dotsboxesaz_b200 import endgame, engine  # noqa: E402


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


def real_actions(L, C):
    cols, plane = C + 1, (L + 1) * (C + 1)
    return [a for a in range(2 * plane) if (a < plane and a % cols < C) or (a >= plane and (a - plane) // cols < L)]


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


def random_states(eng, n, seed, min_plies, max_plies):
    """positions from uniform random games stopped after min_plies .. max_plies plies"""
    gen = torch.Generator(device=eng.device)
    gen.manual_seed(seed)
    depth = torch.randint(min_plies, max_plies + 1, (n,), generator=gen, device=eng.device)
    st = eng.new_states(n)
    for ply in range(max_plies):
        valid = eng.valid_moves(st).double()
        live = (depth > ply) & (eng.result(st) == 2) & (valid.sum(1) > 0)
        mv = torch.multinomial(valid + (valid.sum(1, keepdim=True) == 0).double(), 1, generator=gen).reshape(-1)
        eng.play(st, torch.where(live, mv, torch.full_like(mv, -1)).int())
    return st


def time_launches(fn, reps):
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
    for board in [(5, 5), (7, 7)]:
        eng = engine.Engine(board, n_games=1, max_nodes=16)
        eg = endgame.EndgameSolver(eng, 16)
        for n in (4096, 32768):
            P = torch.empty((n, eng.A), dtype=torch.float32, device=eng.device)
            V = torch.empty((n,), dtype=torch.float32, device=eng.device)
            for f in (4, 8, 10, 12, 14, 16):
                st = mask_states(eng, f, n, seed=f * 100003 + n)
                reps = args.reps if f <= 12 else max(5, args.reps // 10)
                us_eval = time_launches(lambda: eg.evaluate(eng, st, P, V, 0), reps)
                us_moves = time_launches(lambda: eg.moves(st), reps)
                us_fake = time_launches(lambda: eng.fake_nn(st, 0, P, V), args.reps)
                emit(args.out, {"figure": "kernels", "board": "%dx%d" % board, "rows": n, "free_edges": f, "max_free": 16,
                                "k_endgame_eval_us": us_eval, "k_endgame_moves_us": us_moves, "k_fake_nn_us": us_fake,
                                "positions_per_s": n / us_eval * 1e6,
                                "table_updates_per_position": f * 2 ** (f - 1)})
        eng.close()
        torch.cuda.empty_cache()


def bench_search(args):
    n, sims = 16384, 800
    eng = engine.Engine((5, 5), n_games=n, max_nodes=sims + 8, eval_cache=24)
    eng.set_mode(False, 4)
    fake = engine.FakeNetEvaluator(0)
    evs = {"fake": fake,
           "endgame_8": endgame.EndgameEvaluator(fake, endgame.EndgameSolver(eng, 8)),
           "endgame_12": endgame.EndgameEvaluator(fake, endgame.EndgameSolver(eng, 12))}
    rng = np.random.RandomState(1234)
    for name, (lo, hi) in (("roots_0_12", (0, 12)), ("roots_36_44", (36, 44))):
        roots = random_states(eng, n, seed=1234, min_plies=lo, max_plies=hi)
        roots = torch.where((eng.result(roots) == 2).unsqueeze(1), roots, eng.new_states(n)).contiguous()
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
        emit(args.out, {"figure": "search", "board": "5x5", "roots": name, "trees": n, "sims": sims,
                        "sims_per_s": {k: sorted(v) for k, v in res.items()},
                        "median_sims_per_s": {k: float(np.median(v)) for k, v in res.items()}, "device_loop": eng.device_loop,
                        "errors": info["errors"]})
    eng.close()


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=100, help="timed launches per kernel figure (a tenth for f >= 14)")
    ap.add_argument("--rounds", type=int, default=3, help="alternating timed searches per evaluator")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    ap.add_argument("--only", default="kernels,search")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("endgame_bench.py measures the GPU kernels: no CUDA device")
    emit(args.out, {"figure": "gpu", "gpu": gpu_info()})
    parts = args.only.split(",")
    if "kernels" in parts:
        bench_kernels(args)
    if "search" in parts:
        bench_search(args)


if __name__ == "__main__":
    main()
