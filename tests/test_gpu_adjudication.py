"""GPU: adjudication of self-play games with the exact endgame solver (k_selfplay_adjudicate in csrc/dbaz_selfplay.cuh,
BatchedSelfPlay(adjudicate=max_free)).  The kernel alone against EndgameSolver, the 32-edge table and endgame_numpy;
every self-play path against the same games played without adjudication (a prefix of them, cut at the first root with
f <= max_free, with exact z); adjudicate = 0 as a byte-identical control; start states that are solvable already, a
padded chunk and a coach generation."""
import copy
import ctypes

import numpy as np
import pytest

import endgame_ref
from test_gpu_endgame import _rollout_states, _states_by_free

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def mods():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from dotsboxesaz_b200 import endgame, engine, self_play, solver
    from oracle import solver_ref
    return engine, solver, endgame, self_play, solver_ref


def _bufs(eng, searching, moves, reads, left):
    """dbaz_selfplay_buffers with the four arrays k_selfplay_adjudicate uses and one-move dummies for the rest"""
    from dotsboxesaz_b200._capi import SelfplayBuffers
    n, A, dev = eng.n_games, eng.A, eng.device
    keep = [torch.zeros((n, 8 * A + 64), dtype=torch.float64, device=dev) for _ in range(4)]
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    d = [p(t) for t in keep]
    b = SelfplayBuffers(n_moves=1, inv_temp=d[0], uniforms=d[0], noise=None, reads_by_k=d[0], searching=p(searching),
                        move_idx=d[1], moves=p(moves), h_states=d[2], h_visits=d[2], h_active=d[3], h_moves=d[3], h_stats=d[3],
                        h_q=d[3], noise_buf=d[1], reads=p(reads), left=p(left))
    return b, keep


def _host_margin(g, st_np, r):
    edges = int(st_np["edges"][r][0]) | (int(st_np["edges"][r][1]) << 64)
    btc2 = (int(st_np["btc2"][r][0]), int(st_np["btc2"][r][1]))
    return endgame_ref.endgame_moves(g, edges, btc2, int(st_np["to_play"][r]))[1]


@pytest.mark.parametrize("board", [(3, 3), (5, 5), (7, 7), (1, 31)])
def test_kernel_alone(mods, board):
    """Roots at every f = 0 .. 16 (and beyond), trees that qualify mixed with trees that do not (moves = -1, searching =
    0): margin, searching, reads and left change exactly on the qualifying solvable trees, for first = 0 and 1."""
    engine, solver, endgame, _, solver_ref = mods
    per_f = 60 if board == (3, 3) else 3
    probe = engine.Engine(board, n_games=1, max_nodes=16)
    st = _states_by_free(probe, per_f, seed=board[0] * 41 + board[1], f_max=18)
    probe.close()
    n = st.shape[0]
    eng = engine.Engine(board, n_games=n, max_nodes=16)
    eng.reset_roots(st)
    roots = eng.root_states()
    gen = torch.Generator(device=eng.device)
    gen.manual_seed(11)
    f = endgame.EndgameSolver(eng).free_edges(roots)
    table = solver.Solver(eng).solve() if board == (3, 3) else None
    g = solver_ref.Geometry(*board)
    roots_np = eng.states_to_numpy(roots)
    for mf in (0, 10, 12, 16):
        eg = endgame.EndgameSolver(eng, mf)
        want_margin = eg.margin(roots)
        for first in (0, 1):
            searching = torch.randint(0, 2, (n,), generator=gen, device=eng.device).to(torch.int8)
            moves = torch.where(torch.rand((n,), generator=gen, device=eng.device) < 0.3, -1,
                                torch.randint(0, eng.A, (n,), generator=gen, device=eng.device)).int()
            reads = torch.full((n,), 777, dtype=torch.int32, device=eng.device)
            left = torch.full((1,), 100000, dtype=torch.int32, device=eng.device)
            margin = torch.full((n,), 99, dtype=torch.int8, device=eng.device)
            s0, m0 = searching.clone(), moves.clone()
            bufs, keep = _bufs(eng, searching, moves, reads, left)
            eg.adjudicate(bufs, margin, first=bool(first))
            torch.cuda.synchronize()
            q = ((m0 >= 0) | bool(first)) & (s0 == 1)
            hit = q & (f <= mf)
            assert bool(hit.any()) or mf == 0
            assert torch.equal(margin[hit], want_margin[hit]) and bool((margin[~hit] == 99).all()), (mf, first)
            assert torch.equal(searching, torch.where(hit, torch.zeros_like(s0), s0))
            assert torch.equal(reads, torch.where(hit, torch.full_like(reads, -3), torch.full_like(reads, 777)))
            assert torch.equal(moves, m0)
            assert int(left) == 100000 - int(hit.sum())
            if table is not None:
                assert torch.equal(margin[hit], table.margin(roots[hit].contiguous()))
            elif mf in (12, 16):
                for r in torch.nonzero(hit).reshape(-1)[:24].tolist():
                    assert int(margin[r]) == _host_margin(g, roots_np, r), (board, mf, r)
            del keep
    if board == (1, 31):
        assert bool((f <= 16).any()) and bool((roots[:, 1] != 0).any())  # the second edge word was in play
    eng.close()


def test_error_paths(mods):
    engine, _, endgame, self_play, _ = mods
    eng = engine.Engine((3, 3), n_games=4, max_nodes=16)
    z8 = torch.zeros((4,), dtype=torch.int8, device=eng.device)
    z32 = torch.zeros((4,), dtype=torch.int32, device=eng.device)
    bufs, keep = _bufs(eng, z8, z32.clone(), z32.clone(), z32[:1].clone())
    for mf in (17, -1):
        with pytest.raises(engine.EngineError, match=r"dbaz_selfplay_adjudicate: max_free must be in \[0, 16\], got %d" % mf):
            endgame.EndgameSolver(eng, mf).adjudicate(bufs, z8)
    with pytest.raises(engine.EngineError, match="dbaz_selfplay_adjudicate: null margin"):
        endgame.EndgameSolver(eng, 8).adjudicate(bufs, None)
    bufs.left = None
    with pytest.raises(engine.EngineError, match="a required buffer is NULL"):
        endgame.EndgameSolver(eng, 8).adjudicate(bufs, z8)
    for bad in (17, -1):
        with pytest.raises(ValueError, match="adjudicate"):
            self_play.BatchedSelfPlay(eng, engine.FakeNetEvaluator(0), _params(), adjudicate=bad)
    p = _params()
    p.self_play.adjudicate = 6
    assert self_play.BatchedSelfPlay(eng, engine.FakeNetEvaluator(0), p).endgame.max_free == 6
    assert self_play.BatchedSelfPlay(eng, engine.FakeNetEvaluator(0), _params()).endgame is None
    del keep
    eng.close()


def _params(num_read=48, noise=(0.8, 0.25)):
    from dotsboxesaz_b200 import configuration
    p = copy.deepcopy(configuration.simple)
    p.self_play.mcts.mcts_num_read = num_read
    p.self_play.noise = noise
    return p


def _device_games(bsp):
    """per game slot: [(state, visits, move, stats, q) of every recorded row], from the device history"""
    h = bsp._device_hist
    act = torch.stack(h["active"]).cpu().numpy()
    cols = [torch.stack(h[k]).cpu().numpy() for k in ("states", "visits", "moves", "stats", "q")]
    return [[tuple(c[m, g] for c in cols) for m in range(act.shape[0]) if act[m, g]] for g in range(act.shape[1])]


def _host_games(bsp):
    out = {}
    for r in bsp.rows:
        out.setdefault(r["game_idx"], []).append((r["move_idx"], r["move"], r["player"], r["visits"], r["stats"], r["features"]))
    return out


def _same_row(a, b):
    return all(np.array_equal(np.asarray(x), np.asarray(y)) for x, y in zip(a, b))


def _z_by_game(bsp):
    """game slot -> z of its rows, from _rows_from_device (played_games / get_datasets order)"""
    bsp.rows, bsp.played_games = [], []
    bsp._rows_from_device(False)
    out = {}
    for r in bsp.rows:
        out.setdefault(r["game_idx"], []).append((r["player"], r["z"]))
    return out


def _check_device_prefix(eng, eg, off, on, mf):
    """`on` (adjudicated at mf) is `off` cut at its first row with f <= mf, with exact z; every other game equal, z too"""
    g_off, g_on = _device_games(off), _device_games(on)
    z_off, z_on = _z_by_game(off), _z_by_game(on)
    final = on._device_hist["final"]
    margin = on._device_hist["margin"].cpu().numpy()
    n_adj = 0
    for g in range(eng.n_games):
        states = np.stack([r[0] for r in g_off[g]]) if g_off[g] else np.zeros((0, 4), np.int64)
        f = eg.free_edges(torch.from_numpy(states).to(eng.device).contiguous()).cpu().numpy() if len(states) else np.zeros(0)
        cut = int(np.argmax(f <= mf)) if (f <= mf).any() else None
        if cut is None:
            assert margin[g] == -128
            assert len(g_on[g]) == len(g_off[g]) and all(_same_row(a, b) for a, b in zip(g_on[g], g_off[g])), g
            assert z_on.get(g) == z_off.get(g), g
            continue
        n_adj += 1
        assert len(g_on[g]) == cut and all(_same_row(a, b) for a, b in zip(g_on[g], g_off[g][:cut])), (g, cut)
        root = torch.from_numpy(states[cut:cut + 1]).to(eng.device).contiguous()
        assert torch.equal(final[g:g + 1].view(torch.uint8)[:, :22], root.view(torch.uint8)[:, :22])  # edges, btc2, players
        o = int(eg.outcome(root)[0])
        assert margin[g] == int(eg.margin(root)[0])
        tp = int(eng.states_to_numpy(root)["to_play"][0])
        assert [z for _, z in z_on.get(g, [])] == [o if p == tp else -o for p, _ in z_on.get(g, [])], g
    return n_adj


def _evaluator(engine, endgame, eng, kind):
    ev = engine.FakeNetEvaluator(0)
    return ev if kind == "fake" else endgame.EndgameEvaluator(ev, endgame.EndgameSolver(eng, 16))


@pytest.mark.parametrize("path", ["async", "device"])
@pytest.mark.parametrize("board,n,mf", [((3, 3), 256, 12), ((3, 3), 256, 0), ((5, 5), 128, 10)])
@pytest.mark.parametrize("kind", ["fake", "endgame"])
def test_prefix_identity_device_paths(mods, board, n, mf, kind, path):
    engine, _, endgame, self_play, _ = mods
    eng = engine.Engine(board, n_games=n, max_nodes=1024, eval_cache=14)
    ev = _evaluator(engine, endgame, eng, kind)
    eg = endgame.EndgameSolver(eng, 16)
    runs = []
    for adj in (None, mf):
        bsp = self_play.BatchedSelfPlay(eng, ev, _params(), graph_waves=4, pending=1, adaptive=True, adjudicate=adj)
        fn = bsp.play_games_async if path == "async" else bsp.play_games_device
        info = fn(list(range(n)), seed=5)
        runs.append((bsp, info))
    (off, info_off), (on, info_on) = runs
    n_adj = _check_device_prefix(eng, eg, off, on, mf)
    assert info_on["adjudicated"] == n_adj and info_off["adjudicated"] == 0
    if mf == 0:
        assert n_adj == 0 and info_on["sims"] == info_off["sims"]
        for k in ("states", "visits", "active", "moves", "stats", "q"):
            assert all(torch.equal(a, b) for a, b in zip(off._device_hist[k], on._device_hist[k])), k
        for a, b in zip(off.device_samples(), on.device_samples()):
            assert torch.equal(a, b)
    else:
        assert n_adj > 0 and info_on["sims"] < info_off["sims"]
        if board == (5, 5):
            assert n_adj < n  # some games end at a majority first
    eng.close()


@pytest.mark.parametrize("board,n,mf", [((3, 3), 48, 12), ((3, 3), 48, 0), ((5, 5), 24, 10)])
@pytest.mark.parametrize("kind", ["fake", "endgame"])
def test_prefix_identity_host_rng(mods, board, n, mf, kind):
    """play_games (one legacy NumPy stream per game): every game with adjudication is the same game without it, cut at its
    first root with f <= mf, and its rows take z from EndgameSolver.outcome of that root."""
    engine, _, endgame, self_play, _ = mods
    eng = engine.Engine(board, n_games=n, max_nodes=1024, eval_cache=14)
    ev = _evaluator(engine, endgame, eng, kind)
    eg = endgame.EndgameSolver(eng, 16)
    runs = []
    for adj in (None, mf):
        bsp = self_play.BatchedSelfPlay(eng, ev, _params(), graph_waves=4, pending=1, adaptive=True, adjudicate=adj)
        bsp.play_games(list(range(n)), seeds=[1000 + i for i in range(n)])
        runs.append((bsp, eng.root_states()))
    (off, _), (on, final_on) = runs
    h_off, h_on = _host_games(off), _host_games(on)
    z_off = {gi: [r["z"] for r in off.rows if r["game_idx"] == gi] for gi in range(n)}
    z_on = {gi: [r["z"] for r in on.rows if r["game_idx"] == gi] for gi in range(n)}
    n_adj = 0
    for gi in range(n):
        rows = h_off[gi]
        planes = np.stack([r[5] for r in rows])
        f = eg.free_edges(eg.states_from_planes(torch.from_numpy(planes).to(eng.device))).cpu().numpy()
        if not (f <= mf).any():
            assert len(h_on.get(gi, [])) == len(rows) and all(_same_row(a, b) for a, b in zip(h_on[gi], rows))
            assert z_on[gi] == z_off[gi]
            assert on.played_games[gi][1] == off.played_games[gi][1] and on.played_games[gi][3] == off.played_games[gi][3]
            continue
        n_adj += 1
        cut = int(np.argmax(f <= mf))
        got = h_on.get(gi, [])
        assert len(got) == cut and all(_same_row(a, b) for a, b in zip(got, rows[:cut])), (gi, cut)
        root = final_on[gi:gi + 1].contiguous()
        assert np.array_equal(eng.features(root, torch.int16).reshape(-1).cpu().numpy(), planes[cut])
        o = int(eg.outcome(root)[0])
        tp = int(eng.states_to_numpy(root)["to_play"][0])
        assert z_on[gi] == [o if r[2] == tp else -o for r in got]
        assert on.played_games[gi][3] == o and len(on.played_games[gi][1]) == cut
    assert (n_adj > 0) == (mf > 0)
    if mf == 0:
        df_off, df_on = off.get_datasets(0), on.get_datasets(0)
        assert df_off.equals(df_on)
    eng.close()


def _start_states(eng, endgame, mf, solvable_share, seed):
    """3x3 start states with result NONE: a share with f <= mf, the others with f > mf"""
    n = eng.n_games
    gen = torch.Generator(device=eng.device)
    gen.manual_seed(seed)
    deep = _rollout_states(eng, torch.full((16 * n,), 24 - mf, dtype=torch.int64, device=eng.device), gen)
    deep = deep[eng.result(deep) == 2][:n]
    assert deep.shape[0] == n
    shallow = _rollout_states(eng, torch.full((n,), 24 - mf - 4, dtype=torch.int64, device=eng.device), gen)
    k = int(round(solvable_share * n))
    return torch.cat([deep[:k], shallow[k:]]).contiguous()


@pytest.mark.parametrize("share", [1.0, 0.5])
def test_solvable_start_states(mods, share):
    """Start states already solvable: adjudicated before their first search, with no row; the loop ends (left == 0) on
    the asynchronous path; a mix of solvable and unsolvable start states on all three paths."""
    engine, _, endgame, self_play, _ = mods
    n, mf = 64, 10
    eng = engine.Engine((3, 3), n_games=n, max_nodes=1024, eval_cache=14)
    eg = endgame.EndgameSolver(eng, 16)
    start = _start_states(eng, endgame, mf, share, seed=2)
    solv = (eg.free_edges(start) <= mf).cpu().numpy()
    if share == 1.0:
        assert solv.all()
    want = eg.margin(start).cpu().numpy()
    for path in ("async", "device", "host"):
        bsp = self_play.BatchedSelfPlay(eng, engine.FakeNetEvaluator(0), _params(), graph_waves=4, pending=1, adaptive=True,
                                        adjudicate=mf)
        if path == "host":
            info = bsp.play_games(list(range(n)), seeds=list(range(n)), start_states=start.clone())
            rows_of = np.asarray([r["game_idx"] for r in bsp.rows], dtype=np.int64)
            z = {gi: bsp.played_games[gi][3] for gi in range(n)}
        else:
            info = getattr(bsp, "play_games_" + path)(list(range(n)), seed=1, start_states=start.clone())
            assert info["adjudicated"] >= int(solv.sum())
            assert np.array_equal(bsp._device_hist["margin"].cpu().numpy()[solv], want[solv])
            _, _, _, slot, _ = bsp.device_samples()
            rows_of = slot.cpu().numpy()
            z = None
        assert not np.isin(rows_of, np.flatnonzero(solv)).any(), path
        if share == 1.0 and path != "host":
            assert info["sims"] == 0 and len(rows_of) == 0
        if z is not None:
            for gi in np.flatnonzero(solv):
                assert z[gi] == int(np.sign(want[gi]))
    eng.close()


def test_padded_chunk_and_frames_agree(mods):
    """play_shard with a short last chunk (padding games of index -1): no row with f <= max_free, and
    batch_from_selfplay, get_datasets() and played_games agree row for row on z."""
    engine, _, endgame, self_play, _ = mods
    from dotsboxesaz_b200 import samples
    n, mf = 64, 12
    eng = engine.Engine((3, 3), n_games=n, max_nodes=1024, eval_cache=14)
    p = _params()
    p.self_play.adjudicate = mf
    p.self_play.mcts.max_async_searches = 1
    batch, frames, info = self_play.play_shard(p, 0, eng, engine.FakeNetEvaluator(0), list(range(40)), want_frames=True)
    eg = endgame.EndgameSolver(eng, 16)
    f = eg.free_edges(eg.states_from_planes(batch.planes))
    assert len(batch) > 0 and bool((f > mf).all())
    df = frames[0]
    assert len(df) == len(batch) and set(df.index.get_level_values("game_idx")) <= set(range(40))
    meta = batch.meta.cpu().numpy()
    order = np.lexsort((meta[:, 2], meta[:, 1]))
    assert np.array_equal(df["z"].to_numpy().astype(np.float32), batch.z.cpu().numpy()[order])
    # one more chunk by hand: played_games, the DataFrame and the sample batch
    bsp = self_play.BatchedSelfPlay(eng, engine.FakeNetEvaluator(0), p)
    idx = list(range(40)) + [-1] * 24
    info = bsp.play_games_async(idx, seed=9)
    assert info["adjudicated"] > 0
    b = samples.batch_from_selfplay(bsp, 0)
    df = bsp.get_datasets(0, False)
    df = df[df.index.get_level_values("game_idx") >= 0]
    m = b.meta.cpu().numpy()
    order = np.lexsort((m[:, 2], m[:, 1]))
    assert np.array_equal(df["z"].to_numpy().astype(np.float32), b.z.cpu().numpy()[order])
    bsp._rows_from_device(False)
    rz = np.asarray([r["z"] for r in bsp.rows if r["game_idx"] >= 0], dtype=np.float32)
    assert np.array_equal(rz, df["z"].to_numpy().astype(np.float32))
    for gi, mv, vis, z in bsp.played_games:
        if gi >= 0:
            zs = df.xs(gi, level="game_idx")["z"].to_numpy()
            pl = df.xs(gi, level="game_idx")["player"].to_numpy()
            assert len(vis) == len(zs) and set(np.abs(zs)) <= {abs(z)}
            assert len(set(zip(pl, zs))) <= 2
    eng.close()


def test_coach_generation(mods, tmp_path):
    """One learn_to_play generation on 3x3 with adjudication on: every exported row has f > max_free."""
    engine, _, endgame, _, _ = mods
    from dotsboxesaz_b200 import coach, configuration
    from dotsboxesaz_b200.dots_boxes.dots_boxes_game import BoxesState
    from dotsboxesaz_b200.utils.utils import ReplayStore
    BoxesState.init_static_fields(((3, 3),))
    params = copy.deepcopy(configuration.simple)
    for key, name in (("data_root", ""), ("hdf_file", "sp_data"), ("tensorboard_log", "tboard")):
        params[key] = str(tmp_path / name)
    params.elo.hdf_file = str(tmp_path / "elo_data")
    params.nn.chkpts_filename = str(tmp_path / "model_gen{}.pt")
    params.self_play.num_games = 64
    params.self_play.concurrent_games = 64
    params.self_play.max_nodes_per_tree = 1024
    params.self_play.mcts.mcts_num_read = 50
    params.self_play.adjudicate = 12
    params.self_play.export_frames = True
    params.nn.pytorch_device = "cuda:0"
    params.nn.train_params.nb_epochs = 1
    params.nn.train_params.train_batch_size = 256
    params.nn.train_params.val_batch_size = 64
    timings = coach.learn_to_play(params, 0, 0)
    data = ReplayStore(params.hdf_file).read("fresh")
    assert len(data) == timings[0]["rows"] > 0
    eng = engine.Engine((3, 3), n_games=1, max_nodes=16)
    eg = endgame.EndgameSolver(eng, 16)
    x = data[[c for c in data.columns if c.startswith("x_")]].to_numpy().astype(np.int16)
    f = eg.free_edges(eg.states_from_planes(torch.from_numpy(x))).cpu().numpy()
    assert (f > 12).all()
    eng.close()
