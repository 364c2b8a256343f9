#!/usr/bin/env python
"""bench.py -- MCTS simulations/sec of the self-play hot path (BASELINE.json metric).

Own arm (default):   python bench.py --gpus N --steps K --warmup W
Reference arm:       python bench.py --impl reference --gpus N --steps K --warmup W

A "step" is one UCT_search (`--sims` simulations per tree, default 800) for every one of the
`--games` concurrent games of a GPU (default 4096, 3x3 boxes = BASELINE configs[1]) from synthetic
root positions, with Dirichlet root noise (0.8, 0.25) and the reference's SimpleNN (random-init,
seed 0) as leaf evaluator.  One process per GPU; games are sharded by index, there is no data-path
collective (weak scaling).  Rank 0 prints ONE JSON line (stdout carries nothing else).
`--dump-outputs DIR` also writes what the last timed step computed as .npy files; the inputs are seeded, so two builds
run with the same arguments can be compared output for output.

The engine's eval cache (the reference's LRU of net outputs, utils/proxies.py:23-26) is part of the path and is
EMPTIED at the start of every step, inside the timed region.  Keys of the line beyond the contract:
  roofline       k_search_step against the HBM roofline (algorithmic bytes per simulation x simulations per launch /
                 mean launch duration, CUDA events around every launch with the real evaluator in between)
  roofline_net   the evaluator at full width against the sustained bf16 tensor peak
  cpu_baseline   the real reference (oracle/_ref, staged by oracle/make_ref.sh; oracle/py_port.py if absent) on the host cores, bounded sample (N=1 only)
  ablation       the same step with the eval cache switched off, and whether the visit counts agree
  selfplay       whole self-play games per hour (`--selfplay-games` concurrent games per GPU, samples to the host)
  configs        (N = 1) bounded sub-runs of BASELINE's other configurations and modes: configs[2] (5x5 x 2^20 random
                 rollouts, plies/s), configs[3] (5x5 x 16384 games x 800 sims, ResNetZero bf16 with the tcgen05 tower
                 kernel), max_pending_evals = 64 (the reference's shipped mode), SimpleNN in IEEE fp32 and TF32
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "mcts_sims_per_sec"
UNIT = "sims/s"
NOISE = (0.8, 0.25)
MAX_ROOT_PLIES = 12


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--board", default="3x3")
    ap.add_argument("--games", type=int, default=4096, help="concurrent games per GPU")
    ap.add_argument("--sims", type=int, default=800, help="simulations per move")
    ap.add_argument("--net", default="simple", choices=["simple", "resnet", "fake"])
    ap.add_argument("--net-dtype", default="bf16", choices=["bf16", "fp16", "fp32"])
    ap.add_argument("--net-plan", default="fused", choices=["fused", "module"],
                    help="fused: library convs/GEMMs + the engine's fused epilogue kernels; module: the plain nn.Module")
    ap.add_argument("--no-tower", action="store_true", help="ResNetZero: library (cuDNN) convolutions instead of the tcgen05 tower kernel")
    ap.add_argument("--graph-waves", type=int, default=8)
    ap.add_argument("--pending", type=int, default=1,
                    help="max_pending_evals: simulations in flight per tree (1 = strictly sequential, BASELINE configs[1]; "
                         "the reference ships 64, configuration.py:35)")
    ap.add_argument("--eval-cache", type=int, default=24,
                    help="log2(entries) of the device eval cache (the reference's LRU of net outputs, utils/proxies.py:23-26); "
                         "emptied at the start of EVERY step, inside the timed region; 0 = off")
    ap.add_argument("--no-adaptive", action="store_true", help="fixed number of full-width waves instead of the adaptive loop")
    ap.add_argument("--max-inline", type=int, default=4, help="bound on simulations per tree and wave finished without the net "
                                                              "(by count; the captured wave loops bound them by time, --chain-us)")
    ap.add_argument("--chain-us", type=int, default=-1, help="time bound of the in-kernel chains in microseconds (0 = by count only; "
                                                             "-1 = the engine's default, 20)")
    ap.add_argument("--ladder-steps", type=int, default=16, help="evaluator batch sizes of the adaptive loop: games * k / steps")
    ap.add_argument("--no-ablation", action="store_true", help="skip the extra no-cache measurement")
    ap.add_argument("--no-selfplay", action="store_true", help="skip the games/hour measurement (whole self-play games)")
    ap.add_argument("--selfplay-nodes", type=int, default=4096, help="node pool per tree of the self-play engine (tree reuse)")
    ap.add_argument("--selfplay-mode", default="async", choices=["async", "lockstep"],
                    help="async: every game at its own pace (BatchedSelfPlay.play_games_async); lockstep: all games move together")
    ap.add_argument("--selfplay-eval-cache", type=int, default=-1,
                    help="log2(entries) of the self-play engine's eval cache; -1 = sized for the engine "
                         "(self_play.eval_cache_log2_for: 2^27 entries for 32768 games of 3x3 on a B200)")
    ap.add_argument("--selfplay-games", type=int, default=32768,
                    help="concurrent games per GPU of the games/hour measurement (the sims/s workload stays at --games)")
    ap.add_argument("--no-configs", action="store_true",
                    help="skip the `configs` key: BASELINE configs[2] (5x5 random rollouts), configs[3] (5x5 x 16384 x 800, ResNetZero), "
                         "the max_pending_evals = 64 mode and the fp32 / TF32 nets (bounded sub-runs, N = 1 only)")
    ap.add_argument("--tf32", action="store_true", help="with --net-dtype fp32: allow TF32 tensor-core math (off: IEEE fp32)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-workers", type=int, default=0, help="processes for the CPU baseline (0 = min(cores-1, 64))")
    ap.add_argument("--cpu-positions", type=int, default=2, help="searches per worker in the bounded CPU sample")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (root visits, W and priors of every game; the end-to-end "
                         "arm's visits) to DIR/<name>.npy, float32/float64, at most 64 MB in all")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    return args


def workload_name(args):
    return ("%s boxes, %d concurrent games/GPU, %d sims/move, one UCT_search per step from synthetic roots "
            "(0-%d random plies), Dirichlet%s, net=%s" % (args.board, args.games, args.sims, MAX_ROOT_PLIES, NOISE, args.net))


# ------------------------------------------------------------------ CPU side
def cpu_workers(args):
    cores = os.cpu_count() or 1
    return args.cpu_workers if args.cpu_workers > 0 else max(1, min(cores - 1, 64))


def cpu_impl():
    """("reference", oracle.ref_driver) when the real reference has been staged in oracle/_ref (oracle/make_ref.sh; it
    travels to the GPU box with the snapshot), else ("port", oracle.py_port), the Python restatement."""
    from oracle import ref_driver
    if ref_driver.available():
        return "reference", ref_driver
    from oracle import py_port
    return "port", py_port


def cpu_impl_text(kind):
    if kind == "reference":
        return ("the UNMODIFIED reference (oracle/_ref = /root/reference staged by oracle/make_ref.sh): mcts.UCT_search + "
                "utils.proxies.AsyncBatchedProxy(48, 50 ms, 400k LRU) + nn.NeuralNetWrapper + SimpleNN fp32 on CPU, "
                "max_pending_evals 64, 1 torch thread per process")
    return ("oracle/py_port.py (Python/NumPy restatement of the reference incl. its 48-batch/50 ms proxy and 400k LRU, SimpleNN "
            "fp32 on CPU, 1 torch thread per process)")


def run_cpu_sample(args, pool, workers, n_pos, seed0):
    """Every worker runs `n_pos` searches of the bench workload on the reference's own code (or, where oracle/_ref is
    missing, on its Python restatement): asyncio MCTS + age-triggered batching proxy + SimpleNN on CPU, 1 torch thread
    per process -- the reference's own process layout, self_play.py:291-306."""
    _, impl = cpu_impl()
    L, C = (int(x) for x in args.board.split("x"))
    net = "simple" if args.net != "fake" else "fake"
    jobs = [((L, C), args.sims, n_pos, seed0 + w, net, MAX_ROOT_PLIES) for w in range(workers)]
    t0 = time.time()
    res = pool.map(impl.worker_search, jobs)
    wall = time.time() - t0
    sims = sum(r[0] for r in res)
    return sims, wall


def cpu_baseline(args):
    import multiprocessing as mp
    workers = cpu_workers(args)
    ctx = mp.get_context("spawn")
    with ctx.Pool(workers) as pool:
        run_cpu_sample(args, pool, workers, 1, 1000)  # warm-up: imports, torch init
        sims, wall = run_cpu_sample(args, pool, workers, args.cpu_positions, 2000)
    kind = cpu_impl()[0]
    extra = {}
    if kind == "reference":
        # BASELINE configs[0] (the reference's own CPU-runnable case) and its tree-only rate, one process each
        from oracle import ref_driver
        L, C = (int(x) for x in args.board.split("x"))
        try:
            with ctx.Pool(2) as pool:
                game = pool.apply_async(ref_driver.worker_game, ((((L, C)), 100, 1, 0, "simple"),))
                tree = pool.apply_async(ref_driver.worker_search, (((L, C), args.sims, 2, 7, "fake", MAX_ROOT_PLIES),))
                gs, gdt, gn, gmoves = game.get(timeout=600)
                ts, tdt = tree.get(timeout=600)
            extra = {"configs0_reference_1game_100sims": {"value": gs / gdt, "unit": UNIT, "cores": 1, "games_per_hour": gn / gdt * 3600.0,
                                                           "sample": "%d game(s) of %d moves, %d sims in %.1f s: SelfPlay.play_game of the reference, SimpleNN fp32 "
                                                                     "on CPU behind AsyncBatchedProxy, 100 sims/move (BASELINE configs[0])" % (gn, gmoves, gs, gdt)},
                     "tree_only_fake_net": {"value": ts / tdt, "unit": UNIT, "cores": 1,
                                            "sample": "2 x UCT_search(%d) of the reference with the deterministic fake net (no NN, no proxy), 1 process" % args.sims}}
        except Exception as e:  # noqa: BLE001
            extra = {"configs0_reference_1game_100sims": {"error": repr(e)}}
    return {**extra, "value": sims / wall, "unit": UNIT, "cores": workers, "kind": kind,
            "sample": "%d processes x %d UCT_search(%d sims) of the bench workload on %s; %d sims in %.1f s wall"
                      % (workers, args.cpu_positions, args.sims, cpu_impl_text(kind), sims, wall),
            "host_cores": os.cpu_count()}


def c_oracle_rate(args):
    """Single-core rate of the C oracle (fake net, tree-only) -- context for the port's number."""
    from oracle import oracle
    L, C = (int(x) for x in args.board.split("x"))
    t0 = time.time()
    _, _, sims, _ = oracle.selfplay_argmax(L, C, args.sims)
    return sims / (time.time() - t0)


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    workers = cpu_workers(args)
    ctx = mp.get_context("spawn")
    per_step = 1
    with ctx.Pool(workers) as pool:
        for w in range(max(args.warmup, 1)):
            run_cpu_sample(args, pool, workers, per_step, 100 + 1000 * w)
        tot_sims, tot_wall = 0, 0.0
        for k in range(args.steps):
            s, wl = run_cpu_sample(args, pool, workers, per_step, 50000 + 1000 * k)
            tot_sims += s
            tot_wall += wl
    value = tot_sims / tot_wall
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1000.0 * tot_wall / max(args.steps, 1), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64 PUCT over f32/i32 node stats (NumPy); net fp32 on CPU", "data": "synthetic",
            "impl": "reference",
            "config": {"workload": workload_name(args), "board": args.board, "sims_per_move": args.sims,
                       "step": "each of %d processes runs %d UCT_search(%d) on a synthetic root" % (workers, per_step, args.sims)},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": workers, "kind": cpu_impl()[0],
                             "sample": "%s; %d processes" % (cpu_impl_text(cpu_impl()[0]), workers), "host_cores": os.cpu_count()},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


# ------------------------------------------------------------------ GPU side
class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.thread.join(timeout=2)
        sm = sorted(float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 7 and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def synthetic_roots(eng, torch, seed):
    """Random legal positions 0..MAX_ROOT_PLIES plies deep, built on the device with the engine's own
    rules kernels (never terminal on 3x3/5x5 at this depth)."""
    g = torch.Generator(device=eng.device)
    g.manual_seed(seed)
    n = eng.n_games
    st = eng.new_states(n)
    depth = torch.randint(0, MAX_ROOT_PLIES + 1, (n,), generator=g, device=eng.device)
    for ply in range(MAX_ROOT_PLIES):
        legal = eng.valid_moves(st).float()
        mv = torch.multinomial(legal + 1e-9, 1, generator=g).reshape(-1).int()
        mv = torch.where((depth > ply) & (legal.sum(1) > 0), mv, torch.full_like(mv, -1))
        eng.play(st, mv)
    return st


def host_noise(rs, valid_np, alpha):
    import numpy as np
    A = valid_np.shape[1]
    return rs.dirichlet(np.ones(A) * alpha, size=valid_np.shape[0]) * valid_np  # mcts.py:220-223


def dump_outputs(path, arrays, limit=64 << 20):
    """Writes every array as path/<name>.npy.  The arrays share their first axis (the game); when they exceed `limit`
    bytes in all, a fixed seeded sample of games is written instead, the same one in every run with the same arguments."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    n = len(next(iter(arrays.values())))
    total = sum(a.nbytes for a in arrays.values())
    rows = np.arange(n)
    if total > limit:
        rows = np.sort(np.random.RandomState(0).choice(n, n * limit // total, replace=False))
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a[rows])


def sub_bench(extra, timeout=420):
    """One bounded sub-run of this script (its own process: its own engine, graphs and HBM), parsed JSON line or error."""
    cmd = [sys.executable, os.path.abspath(__file__), "--gpus", "1", "--no-cpu-baseline", "--no-ablation", "--no-selfplay",
           "--no-configs"] + extra
    env = dict(os.environ)
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    try:
        out = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=timeout, env=env, text=True)
        lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
        if out.returncode != 0 or not lines:
            return {"error": "rc=%d %s" % (out.returncode, out.stderr[-300:])}
        return json.loads(lines[-1])
    except Exception as e:  # noqa: BLE001 -- a failed sub-run must not lose the main line
        return {"error": repr(e)}


def pick(d, roof_keys=("kernel", "achieved", "peak", "unit", "frac", "kernel_us", "share_of_step", "algorithmic_bytes_per_sim",
                       "sims_per_launch", "launches_per_step", "cache_hit_frac", "terminal_leaf_frac", "mean_path_nodes")):
    """The part of a sub-run's line the `configs` key keeps."""
    if "error" in d:
        return d
    out = {k: d.get(k) for k in ("metric", "value", "unit", "ms_per_step", "steps", "warmup", "gpu_launches", "dtype")}
    out["e2e"] = (d.get("e2e") or {}).get("value")
    out["workload"] = (d.get("config") or {}).get("workload")
    if d.get("roofline"):
        out["roofline"] = {k: d["roofline"].get(k) for k in roof_keys}
    if d.get("roofline_net"):
        out["roofline_net"] = {k: d["roofline_net"].get(k) for k in ("kernel", "achieved", "peak", "unit", "frac", "us_per_batch")}
    return out


def rollout_config(torch, dev, n=1 << 20, board=(5, 5)):
    """BASELINE configs[2]: uniformly random legal playouts of `n` concurrent 5x5 games to the end (Philox4x32-10, one
    thread per game, the whole game in registers).  plies/s with CUDA events over 5 launches on fresh states; the HBM
    figure uses SURVEY 8d's 32 bytes per ply -- the kernel is bound by integer issue, not by HBM (profiles/)."""
    from dotsboxesaz_b200 import engine
    eng = engine.Engine(board, n_games=8, max_nodes=16, device=dev)
    try:
        fresh = eng.new_states(n)
        st = fresh.clone()
        plies = eng.random_rollout(st, seed=0)
        torch.cuda.synchronize()
        total = int(plies.sum())
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ms = 0.0
        reps = 5
        for r in range(reps):
            st.copy_(fresh)
            a.record()
            eng.random_rollout(st, seed=0)
            b.record()
            torch.cuda.synchronize()
            ms += a.elapsed_time(b)
        sec = ms / reps / 1e3
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        gbs = total * 32 / sec / 1e9
        # host-to-host: packed states from pinned memory, final states and ply counts back
        host_in = fresh.cpu().pin_memory()
        host_out = torch.empty_like(host_in).pin_memory()
        plies_out = torch.empty((n,), dtype=torch.int32).pin_memory()
        t0 = time.time()
        st.copy_(host_in, non_blocking=True)
        pl = eng.random_rollout(st, seed=0)
        host_out.copy_(st, non_blocking=True)
        plies_out.copy_(pl, non_blocking=True)
        torch.cuda.synchronize()
        e2e_sec = time.time() - t0
        out = {"metric": "random_rollout_plies_per_sec", "value": total / sec, "unit": "plies/s", "games_per_sec": n / sec,
               "games": n, "plies_per_game": total / n, "ms_per_launch": sec * 1e3, "gpu_launches": 1,
               "e2e": total / e2e_sec, "e2e_h2d_d2h_bytes": int(host_in.numel() * 8 * 2 + n * 4),
               "workload": "%dx%d boxes, %d concurrent games, uniformly random legal moves to the end (BASELINE configs[2])" % (board[0], board[1], n),
               "roofline": {"bound": "hbm", "kernel": "k_game_rollout", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak,
                            "algorithmic_bytes_per_ply": 32, "note": "one thread plays a whole game in registers, HBM sees each state once in and once out: the algorithmic 32 bytes per ply are SURVEY 8d's accounting, the DRAM traffic is far below it"}}
    finally:
        eng.close()
    # the reference's BoxesState on one host core, bounded sample
    try:
        kind, impl = cpu_impl()
        if kind == "reference":
            p, sec_cpu = impl.worker_rollouts((board, 200, 0))
            out["cpu_baseline"] = {"value": p / sec_cpu, "unit": "plies/s", "cores": 1, "kind": "reference",
                                   "sample": "200 random 5x5 playouts with the reference's BoxesState.play_ (oracle/_ref), 1 process"}
    except Exception as e:  # noqa: BLE001
        out["cpu_baseline"] = {"error": repr(e)}
    return out


def coach_config(args, torch, dist, rank, world, dev, board=(5, 5), games_per_rank=1024, sims=200):
    """BASELINE configs[4]: full coach iterations (self-play + NCCL sample gather + train + NCCL weight broadcast), 5x5,
    ResNetZero (20 blocks), games sharded over the ranks.  Generations 0 and 1 (generation 0 trains 0 epochs -- the
    reference's min(2 * generation, nb_epochs), nn.py:205 -- generation 1 trains one).  Bounded: 1024 games per rank at
    200 sims/move, at most 65536 training positions."""
    import copy
    import tempfile
    import shutil
    from dotsboxesaz_b200 import coach, configuration
    from dotsboxesaz_b200.dots_boxes.dots_boxes_game import BoxesState
    from dotsboxesaz_b200.nn import resnet_zero_parameters
    BoxesState.init_static_fields((board,))
    params = copy.deepcopy(configuration.resnet)
    params.nn.model_parameters = resnet_zero_parameters(board, nb_blocks=20)
    root = tempfile.mkdtemp(prefix="dbaz_coach_") if rank == 0 else None
    box = [root]
    dist.broadcast_object_list(box, src=0)
    root = box[0]
    params.rewrite_str("data/_exp_", root)
    params.self_play.num_games = games_per_rank * world
    params.self_play.concurrent_games = games_per_rank
    params.self_play.max_nodes_per_tree = 4096
    params.self_play.mcts.mcts_num_read = sims
    params.self_play.export_frames = False
    params.nn.pytorch_device = "cuda:%d" % torch.cuda.current_device()
    params.nn.train_params.nb_epochs = 1
    params.nn.train_params.train_batch_size = 1024
    params.nn.train_params.val_batch_size = 1024
    params.nn.train_params.max_samples_per_gen = 65536
    t0 = time.time()
    tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = True  # PyTorch's default, i.e. what the reference's fp32 training runs with (the search part of this file switches it off)
    try:
        timings = coach.learn_to_play(params, 0, 1)
    finally:
        torch.backends.cudnn.allow_tf32 = tf32
        BoxesState.init_static_fields(((3, 3),))
        if rank == 0:
            shutil.rmtree(root, ignore_errors=True)
    if rank != 0:
        return None
    g1 = timings[-1]
    return {"workload": "%dx%d boxes, ResNetZero 20 blocks bf16, %d games/generation (%d per GPU) at %d sims/move, generations 0-1, "
                        "samples gathered with NCCL, rank 0 trains, weights broadcast with NCCL (BASELINE configs[4])"
                        % (board[0], board[1], games_per_rank * world, games_per_rank, sims),
            "n_gpus": world, "total_s": time.time() - t0, "generations": timings,
            "selfplay_games_per_hour": games_per_rank * world / max(g1.get("play_s", 1e-9), 1e-9) * 3600.0,
            "gather_s": g1.get("gather_s"), "train_s": g1.get("train_s"), "broadcast_s": g1.get("broadcast_s"), "rows": g1.get("rows")}


def other_configs(args, torch, dev):
    """BASELINE.json configs beyond the headline and the modes the verdict asked for, each as a bounded sub-run."""
    out = {}
    try:
        out["configs2_rollouts_5x5_1M"] = rollout_config(torch, dev)
    except Exception as e:  # noqa: BLE001
        out["configs2_rollouts_5x5_1M"] = {"error": repr(e)}
    torch.cuda.empty_cache()
    out["configs3_5x5_16384games_800sims_resnet_bf16"] = pick(sub_bench(
        ["--board", "5x5", "--net", "resnet", "--games", "16384", "--sims", "800", "--steps", "2", "--warmup", "3", "--eval-cache", "22"]))
    out["max_pending_evals_64_3x3_4096games"] = pick(sub_bench(
        ["--board", "3x3", "--net", "simple", "--games", "4096", "--sims", "800", "--pending", "64", "--steps", "2", "--warmup", "3"]))
    out["net_fp32_ieee_3x3_4096games"] = pick(sub_bench(
        ["--board", "3x3", "--net", "simple", "--games", "4096", "--sims", "800", "--net-dtype", "fp32", "--steps", "1", "--warmup", "3"]))
    out["net_tf32_3x3_4096games"] = pick(sub_bench(
        ["--board", "3x3", "--net", "simple", "--games", "4096", "--sims", "800", "--net-dtype", "fp32", "--tf32", "--steps", "1", "--warmup", "3"]))
    return out


_REAL_STDOUT = None


def claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries print there too (NCCL's version banner when NCCL_DEBUG is set
    in the environment), so fd 1 is pointed at stderr for the whole run and the JSON line goes to the saved descriptor."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    args = parse_args()
    claim_stdout()
    if args.impl == "reference":
        reference_arm(args)
        return

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # NCCL's version banner must not share stdout with the JSON line

    # CPU baseline first (rank 0, N=1 only), before CUDA is initialised, so the two never overlap
    cpu = None
    c_rate = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline(args)
        c_rate = c_oracle_rate(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    from dotsboxesaz_b200 import engine
    from dotsboxesaz_b200.nn import (DeviceEvaluator, FusedResNetZero, FusedSimpleNN, ResNetZero, resnet_zero_parameters)
    from dotsboxesaz_b200.dots_boxes.dots_boxes_nn import SimpleNN
    from dotsboxesaz_b200.utils.utils import DotDict

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    torch.backends.cudnn.allow_tf32 = bool(args.tf32)
    torch.backends.cuda.matmul.allow_tf32 = bool(args.tf32)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    L, C = (int(x) for x in args.board.split("x"))
    use_cache = args.eval_cache if args.pending == 1 else 0
    adaptive = (not args.no_adaptive) and args.pending == 1 and args.graph_waves > 0
    eng = engine.Engine((L, C), n_games=args.games, max_nodes=args.sims + 8, device=dev, max_pending=args.pending,
                        eval_cache=use_cache)
    eng.set_mode(False, args.max_inline)
    if args.chain_us >= 0:
        eng.chain_us = args.chain_us
    eng.LADDER_STEPS = args.ladder_steps
    dt = {"bf16": torch.bfloat16, "fp16": torch.float16, "fp32": torch.float32}[args.net_dtype]
    if args.net == "fake":
        ev = engine.FakeNetEvaluator(0)
    else:
        torch.manual_seed(0)
        model = SimpleNN(board=(L, C)) if args.net == "simple" else ResNetZero(
            DotDict({"nn": {"model_parameters": resnet_zero_parameters((L, C))}}))
        if args.net_plan == "fused":
            ev = FusedSimpleNN(model, eng, dtype=dt) if args.net == "simple" else FusedResNetZero(model, eng, dtype=dt, use_tower=not args.no_tower)
        else:
            ev = DeviceEvaluator(model, eng, dtype=dt, channels_last=True)

    eng_chain_us = int(eng.chain_us)
    roots = synthetic_roots(eng, torch, seed=1234 + rank)
    valid_np = eng.valid_moves(roots).cpu().numpy()
    rs = np.random.RandomState(99 + rank)
    noise_dev = torch.from_numpy(host_noise(rs, valid_np, NOISE[0])).to(dev)
    visits = torch.empty((args.games, eng.A), dtype=torch.int32, device=dev)

    def search():
        eng.clear_eval_cache()  # every step starts with an empty table: only reuse within the step's own searches counts
        eng.run_search(args.sims, ev, noise=noise_dev, coeff=NOISE[1], graph_waves=args.graph_waves, pending=args.pending,
                       adaptive=adaptive)

    def step_resident():
        eng.reset_roots(roots)
        search()
        visits.copy_(eng.root_visits())

    # host buffers of the end-to-end arm (pinned)
    roots_host = roots.cpu().pin_memory()
    visits_host = torch.empty((args.games, eng.A), dtype=torch.int32).pin_memory()
    roots_in = torch.empty_like(roots)

    # the end-to-end arm's inputs live in pinned host memory before the clock starts: root states and one host-drawn
    # Dirichlet sample per step (legacy NumPy RNG, as the reference draws it)
    noise_pool = [torch.from_numpy(host_noise(rs, valid_np, NOISE[0])).pin_memory() for _ in range(args.steps + 2)]
    e2e_calls = [0]

    def step_e2e():
        noise_host = noise_pool[e2e_calls[0] % len(noise_pool)]
        e2e_calls[0] += 1
        roots_in.copy_(roots_host, non_blocking=True)
        noise_dev.copy_(noise_host, non_blocking=True)
        eng.reset_roots(roots_in)
        search()
        visits_host.copy_(eng.root_visits(), non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return int(visits_host[0].sum())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.time()
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1), (time.time() - t0) * 1e3], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms[0]), float(ms[1])

    for _ in range(max(args.warmup, 3)):
        step_resident()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    l0, w0 = eng.n_launches, eng.n_waves
    ms, _wall = timed(step_resident, args.steps)
    launches = eng.n_launches - l0
    waves_per_step = (eng.n_waves - w0) / args.steps
    st = eng.status()  # also checks that no tree faulted
    outputs = None
    if args.dump_outputs:  # the trees of the last timed step, read before anything else runs on the engine
        W, P, _, _ = eng.root_children()
        outputs = {"root_visits": visits.float().cpu().numpy(), "root_W": W.cpu().numpy(), "root_priors": P.cpu().numpy()}
    for _ in range(2):
        step_e2e()
    ms_e2e, wall_e2e = timed(step_e2e, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    if outputs is not None:
        outputs["e2e_root_visits"] = visits_host.float().numpy()
        dump_outputs(args.dump_outputs, {(k if world == 1 else "%s_rank%d" % (k, rank)): v for k, v in outputs.items()},
                     limit=(64 << 20) // world)

    sims_per_step = args.games * args.sims * world
    value = sims_per_step * args.steps / (ms / 1e3)
    e2e_value = sims_per_step * args.steps / (max(ms_e2e, wall_e2e) / 1e3)

    # ---- roofline of the dominant kernel of MY code (k_search_step), timed live with CUDA events on
    # the launching stream, one event pair per launch, with the real evaluator between launches
    P = st["path_nodes"] / max(1, st["sims"])
    f_term = st["terminal_leaves"] / max(1, st["sims"])
    f_hit = st["cache_hits"] / max(1, st["sims"])
    f_miss = 1.0 - f_term - f_hit  # simulations whose leaf the net evaluated
    A, F = eng.A, eng.F
    plane_b = 4 if (args.net == "fake" or args.net_dtype == "fp32") else 2
    # DESIGN.md section 3: select + leaf create + backup | expand (node priors out, zeroed stats, value) |
    # features out + net priors in (evaluated leaves only) | eval cache probe (every non-terminal leaf) + insert
    bytes_per_sim = ((P - 1) * (13 * A + 24) + 36 + 24 * P + (1 - f_term) * (13 * A + 4) + f_miss * (F * plane_b + 4 * A)
                     + ((1 - f_term) * 16 * A + f_miss * 16 * A if use_cache else 0))
    roof = None
    ablation = None
    net_roof = None
    if rank == 0:
        eng.reset_roots(roots)
        eng.clear_eval_cache()
        eng.set_mode(adaptive, args.max_inline)
        timed_chains = adaptive and eng.chain_us > 0 and args.max_inline > 0 and args.pending == 1
        if timed_chains:  # the kernel the captured wave loop runs: chains bounded by time, the count only a cap
            eng.set_mode(adaptive, eng.CHAIN_COUNT_CAP)
            eng.set_chain_budget(eng.chain_us)
        eng.begin(args.sims, noise_dev, NOISE[1], pending=args.pending)
        evs = []
        n_waves = 2 + max(0, -(-(args.sims - min(args.pending, eng.A)) // args.pending))
        s0 = eng.status()["sims"]
        w = 0
        while w < n_waves:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); eng.step(); b.record()
            ev(eng)
            evs.append((a, b))
            w += 1
            if adaptive and w % 8 == 0 and eng.wave_counts()[1] == 0:
                break
        eng.step()
        torch.cuda.synchronize()
        if timed_chains:
            eng.set_chain_budget(0)
            eng.set_mode(adaptive, args.max_inline)
        n_run = len(evs)
        evs = evs[min(16, n_run // 4):]
        k_ms = sum(a.elapsed_time(b) for a, b in evs) / len(evs)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        sims_per_launch = (eng.status()["sims"] - s0) / n_run  # simulations one launch processes on average
        achieved = bytes_per_sim * sims_per_launch / (k_ms * 1e-3) / 1e9
        traffic = None
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get("k_search_step_dram_bytes_per_launch")
        except Exception:
            pass
        roof = {"bound": "hbm", "kernel": "k_search_step", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": "measured" if peaks else "fallback",
                "kernel_us": k_ms * 1e3, "algorithmic_bytes_per_sim": bytes_per_sim, "mean_path_nodes": P,
                "terminal_leaf_frac": f_term, "cache_hit_frac": f_hit, "share_of_step": k_ms * waves_per_step / (ms / args.steps),
                "sims_per_launch": sims_per_launch, "launches_per_step": waves_per_step}
        # ---- the evaluator (library tensor-core kernels between the engine's stem and heads kernels) at full width:
        # FLOPs per position from BASELINE.md (torch FlopCounterMode), timed here as a graph of 8 calls
        net_roof = None
        flops_pos = {("simple", "3x3"): 62.9e6, ("resnet", "3x3"): 47.3e6, ("resnet", "5x5"): 106.5e6}.get((args.net, args.board))
        if flops_pos and args.net != "fake":
            # full width -- for an evaluator whose cost is a step function of the batch (the tower kernel's tile waves) the
            # widest batch the wave loop actually runs: the largest multiple of its quantum
            q = int(getattr(ev, "batch_quantum", 0) or 0)
            full = args.games * args.pending  # rows of a full-width wave: one per in-flight simulation
            net_rows = full if (q <= 0 or q > full or args.pending > 1) else (full // q) * q
            eng.pending = args.pending
            eng._batch_rows = None if net_rows == full else net_rows
            for _ in range(3):
                ev(eng)
            torch.cuda.synchronize()
            gnet = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gnet):
                for _ in range(8):
                    ev(eng)
            gnet.replay()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); gnet.replay(); gnet.replay(); b.record()
            torch.cuda.synchronize()
            net_us = a.elapsed_time(b) / 16 * 1e3
            del gnet
            eng._batch_rows = None
            tf = net_rows * flops_pos / net_us / 1e6
            tpeak = float(peaks.get("bf16_tflops_sustained", 1400.0))
            own = "k_nn_stem_mma + k_resnet_tower (tcgen05) + head GEMM (library) + k_nn_heads" if q else "library conv/GEMM kernels + k_nn_stem_mma + k_nn_heads"
            net_roof = {"bound": "tensor", "kernel": "evaluator, %d leaves: %s" % (net_rows, own),
                        "achieved": tf, "peak": tpeak, "unit": "TFLOP/s", "frac": tf / tpeak, "us_per_batch": net_us,
                        "peak_source": "measured, sustained bf16" if peaks else "fallback", "flops_per_position": flops_pos}
        if use_cache and not args.no_ablation and world == 1:
            # the same step (a) with the table switched off (fixed wave loop, row == tree): what the cache buys, and
            # (b) with the table on but every evaluator batch at full width, i.e. at the batch size of (a): the cache and
            # the scheduling change no visit count; the production run (shrinking batches) can differ from (a) only through
            # the library kernels the net picks at another batch size
            step_resident()
            vis_adaptive = visits.clone()
            eng._ladder = lambda evaluator=None: [eng.n_games]
            step_resident()
            vis_full = visits.clone()
            del eng._ladder
            eng.set_eval_cache(0)

            def step_plain():
                eng.reset_roots(roots)
                eng.run_search(args.sims, ev, noise=noise_dev, coeff=NOISE[1], graph_waves=args.graph_waves, pending=args.pending)
                visits.copy_(eng.root_visits())
            step_plain()
            ms_plain, _ = timed(step_plain, 2)
            ablation = {"no_eval_cache_sims_per_sec": args.games * args.sims * 2 / (ms_plain / 1e3),
                        "visit_counts_equal_cached_vs_uncached_at_equal_batch_size": bool((vis_full == visits).all()),
                        "trees_with_identical_visit_counts_production_vs_uncached": float((vis_adaptive == visits).all(1).float().mean())}

    # ---- the other half of BASELINE's metric: whole self-play games per hour.  `games` games per GPU from the empty
    # board to the end (800 sims/move, tree reuse, Dirichlet noise, temperature schedule {0: 1.0, 12: 0.02}), device-
    # resident loop, eval cache emptied before the timed batch; the clock stops when the (planes, pi, z) samples are in
    # host memory.
    selfplay = None
    node_bytes, eng_A = eng.node_bytes, eng.A
    if not args.no_selfplay and args.net != "fake":
        from dotsboxesaz_b200 import self_play as sp_mod
        node_bytes = eng.node_bytes
        eng.close()
        del eng
        torch.cuda.empty_cache()
        # concurrent games: as asked, but the node pools must fit beside the eval cache (80 GB budget)
        sp_nodes = args.selfplay_nodes if eng_A <= 32 else max(args.selfplay_nodes, 6144)
        fit = int(80e9 // (sp_nodes * node_bytes))
        sp_games = max(256, min(args.selfplay_games, fit // 1024 * 1024 if fit >= 1024 else fit))
        sp_cache = use_cache
        if use_cache and args.selfplay_eval_cache != 0:
            sp_cache = (args.selfplay_eval_cache if args.selfplay_eval_cache > 0
                        else max(use_cache, sp_mod.eval_cache_log2_for(eng_A, sp_games, sp_nodes, dev)))
        eng_sp = engine.Engine((L, C), n_games=sp_games, max_nodes=sp_nodes, device=dev, eval_cache=sp_cache)
        eng_sp.set_mode(False, args.max_inline)
        if args.chain_us >= 0:
            eng_sp.chain_us = args.chain_us
        eng_sp.LADDER_STEPS = args.ladder_steps
        if args.net_plan != "fused":
            ev_sp = DeviceEvaluator(model, eng_sp, dtype=dt, channels_last=True)
        elif args.net == "simple":
            ev_sp = FusedSimpleNN(model, eng_sp, dtype=dt)
        else:
            ev_sp = FusedResNetZero(model, eng_sp, dtype=dt, use_tower=not args.no_tower)
        sp_params = DotDict({"self_play": {"reuse_mcts_tree": True, "noise": NOISE,
                                           "mcts": {"mcts_num_read": args.sims, "mcts_cpuct": (1.25, 19652),
                                                    "temperature": {0: 1.0, 12: 0.02}, "max_async_searches": 1}}})
        rows_out = [0]
        pinned = {}

        def play(seed):
            use_async = args.selfplay_mode == "async" and adaptive
            sp = sp_mod.BatchedSelfPlay(eng_sp, ev_sp, sp_params, graph_waves=16 if use_async else args.graph_waves, adaptive=adaptive)
            eng_sp.clear_eval_cache()
            info = (sp.play_games_async if use_async else sp.play_games_device)(range(sp_games), seed=seed)
            outs = sp.device_samples()[:3]  # (planes int16, pi float64, z float32), still on the device
            for k, t in enumerate(outs):     # ... into pinned host buffers (allocated by the warm-up call, reused)
                need = t.numel()
                if k not in pinned or pinned[k].numel() < need:
                    pinned[k] = torch.empty((int(need * 1.1),), dtype=t.dtype).pin_memory()
                pinned[k][:need].copy_(t.reshape(-1), non_blocking=True)
            torch.cuda.current_stream().synchronize()
            rows_out[0] = outs[0].shape[0]
            return info
        play(1000 + rank)  # warm-up: graph captures for this engine
        barrier()
        t0 = time.time()
        info = play(rank)
        barrier()
        sec = torch.tensor([time.time() - t0], dtype=torch.float64, device=dev)
        tot = torch.tensor([float(info["sims"]), float(rows_out[0])], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(sec, op=dist.ReduceOp.MAX)
            dist.all_reduce(tot, op=dist.ReduceOp.SUM)
        selfplay = {"games_per_hour": sp_games * world / float(sec[0]) * 3600.0, "games": sp_games * world,
                    "seconds": float(sec[0]), "sims_per_sec": float(tot[0]) / float(sec[0]), "sample_rows": int(tot[1]),
                    "cache_hit_frac": info["cache_hits"] / max(1, info["sims"]), "eval_cache_log2": int(sp_cache),
                    "terminal_leaf_frac": info["terminal_leaves"] / max(1, info["sims"]),
                    "what": "%d concurrent games per GPU played to the end (%s), tree reuse, temperature {0: 1.0, 12: 0.02}, "
                            "samples copied to the host inside the timed region"
                            % (sp_games, "every game at its own pace" if args.selfplay_mode == "async" and adaptive else "all games move by move")}

    coach_info = None
    if world > 1 and not args.no_configs:
        # BASELINE configs[4]: full coach iterations on N GPUs (every rank takes part)
        for name in ("eng_sp", "eng"):
            obj = locals().get(name)
            if obj is not None:
                try:
                    obj.close()
                except Exception:
                    pass
        torch.cuda.empty_cache()
        try:
            coach_info = coach_config(args, torch, dist, rank, world, dev)
        except Exception as e:  # noqa: BLE001 -- must not lose the main line
            coach_info = {"error": repr(e)}

    configs = None
    if rank == 0 and world == 1 and not args.no_configs:
        # free this process's engines first: the sub-runs need the HBM
        for name in ("eng_sp", "ev_sp", "eng", "ev"):
            obj = locals().get(name)
            if name.startswith("eng") and obj is not None:
                try:
                    obj.close()
                except Exception:
                    pass
        torch.cuda.empty_cache()
        configs = other_configs(args, torch, dev)

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f64 PUCT over f32/i32 node stats; net %s" % (
                    ("tf32" if (args.tf32 and args.net_dtype == "fp32") else args.net_dtype) if args.net != "fake" else "none (fake)"),
                "data": "synthetic",
                "config": {"workload": workload_name(args), "board": args.board, "games_per_gpu": args.games,
                           "sims_per_move": args.sims, "net": args.net, "net_dtype": args.net_dtype, "net_plan": args.net_plan, "max_pending_evals": args.pending,
                           "eval_cache": ("2^%d entries, emptied at the start of every step" % use_cache) if use_cache else "off",
                           "wave_loop": ("adaptive (compact rows, batch ladder, in-kernel chains bounded at %d us)" % eng_chain_us if (adaptive and eng_chain_us > 0)
                                         else "adaptive (compact rows, batch ladder)") if adaptive else "fixed", "parallelism": "games sharded by index x%d, no collective" % world,
                           "l2": "inputs larger than L2: node pool touched per step %.2f GB/GPU vs 126 MB L2" % (
                               args.games * (args.sims + 1) * node_bytes / 1e9),
                           "graph_waves": args.graph_waves},
                "games_per_hour": selfplay["games_per_hour"] if selfplay else None, "selfplay": selfplay,
                "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": max(ms_e2e, wall_e2e) / args.steps,
                        "h2d_bytes_per_step": int(roots_host.numel() * 8 + noise_pool[0].numel() * 8),
                        "d2h_bytes_per_step": int(visits_host.numel() * 4),
                        "api": "Engine.reset_roots(host roots) + Engine.run_search(host Dirichlet noise) + root_visits -> host"},
                "gpu_launches": launches, "roofline": roof, "roofline_net": net_roof, "cpu_baseline": cpu, "clocks": clocks, "ablation": ablation,
                "configs": configs, "coach": coach_info}
        if c_rate is not None:
            line["cpu_c_oracle_1core_sims_per_sec"] = c_rate
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
