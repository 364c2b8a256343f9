"""GPU: exact endgame play in self-play (k_selfplay_exact_endgame in csrc/dbaz_selfplay.cuh,
BatchedSelfPlay(exact_endgame=max_free)).  The kernel alone against EndgameSolver, the 32-edge table, endgame_numpy and a
replay of its draws; every self-play path against the same games played without the mode (equal up to the first root
with f <= max_free, then a legal game of optimal moves to the end, one exact row per ply, with exact z);
exact_endgame = 0 as a byte-identical control; start states that are solvable already, a padded chunk, a coach
generation, grading and the error paths."""
import copy
import ctypes

import numpy as np
import pytest

import endgame_ref
from test_gpu_endgame import _states_by_free
from test_gpu_adjudication import _params, _start_states, _evaluator

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

KINDS = ("outcome", "margin")


@pytest.fixture(scope="module")
def mods():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from dotsboxesaz_b200 import endgame, engine, self_play, solver
    from oracle import solver_ref
    return engine, solver, endgame, self_play, solver_ref


def _draw(vis, u):
    """k_selfplay_pick's draw with weights vis > 0 (all 1): the first action whose running sum exceeds u * total, else the
    last positive weight"""
    w = (vis > 0).double()
    cdf = w.cumsum(1)
    A = vis.shape[1]
    ar = torch.arange(A, device=vis.device)
    first = torch.where(cdf > (u * cdf[:, -1]).unsqueeze(1), ar, A).min(1).values
    last = torch.where(w > 0, ar, -1).max(1).values
    return torch.where(first < A, first, last)


def _published(eng, st):
    """states as a history row holds them: flags 0, depth 0, parent -1, parent_action -1, cached result"""
    out = st.clone()
    v16 = out.view(torch.int16)
    v16[:, 11] = 0
    out.view(torch.int32)[:, 6] = -1
    v16[:, 14] = -1
    v16[:, 15] = eng.result(st).to(torch.int16)
    return out


def _b22(st):
    return st.contiguous().view(torch.uint8).reshape(-1, 32)[:, :22]


class _Buffers:
    """dbaz_selfplay_buffers over real history tables, each filled with a marker so that untouched bytes show"""

    def __init__(self, eng, n_moves, gen):
        from dotsboxesaz_b200._capi import SelfplayBuffers
        n, A, dev = eng.n_games, eng.A, eng.device
        self.t = dict(
            inv_temp=torch.ones((n_moves,), dtype=torch.float64, device=dev),
            uniforms=torch.rand((n_moves, n), dtype=torch.float64, device=dev, generator=gen),
            reads_by_k=torch.ones((A + 1,), dtype=torch.int32, device=dev),
            searching=torch.randint(0, 2, (n,), generator=gen, device=dev).to(torch.int8),
            move_idx=torch.randint(0, 4, (n,), generator=gen, device=dev),
            moves=torch.where(torch.rand((n,), generator=gen, device=dev) < 0.3, -1,
                              torch.randint(0, A, (n,), generator=gen, device=dev)).int(),
            h_states=torch.randint(-2 ** 62, 2 ** 62, (n_moves, n, 4), generator=gen, device=dev),
            h_visits=torch.full((n_moves, n, A), 7, dtype=torch.int32, device=dev),
            h_active=torch.full((n_moves, n), 5, dtype=torch.int8, device=dev),
            h_moves=torch.full((n_moves, n), -9, dtype=torch.int32, device=dev),
            h_stats=torch.full((n_moves, n, 8), 33, dtype=torch.int32, device=dev),
            h_q=torch.full((n_moves, n), 1.5, dtype=torch.float32, device=dev),
            noise_buf=torch.zeros((n, A), dtype=torch.float64, device=dev),
            reads=torch.full((n,), 777, dtype=torch.int32, device=dev),
            left=torch.full((1,), 100000, dtype=torch.int32, device=dev))
        p = lambda x: ctypes.c_void_p(x.data_ptr())
        self.bufs = SelfplayBuffers(n_moves=n_moves, noise=None, **{k: p(v) for k, v in self.t.items()})
        self.t0 = {k: v.clone() for k, v in self.t.items()}


@pytest.mark.parametrize("board", [(3, 3), (5, 5), (7, 7), (1, 31)])
def test_kernel_alone(mods, board):
    """Roots at every f = 0 .. 18, trees that qualify mixed with trees that do not: every solvable qualifying root is
    played out to its first state with a result, one row per ply (the published state, the optimal moves of `kind` as
    visits, zero statistics, the move a replay of the draw gives); exact_margin, searching, reads, move_idx and left
    change exactly as specified, and every other byte of every buffer is left alone."""
    engine, solver, endgame, _, solver_ref = mods
    per_f = 8 if board == (3, 3) else 3
    probe = engine.Engine(board, n_games=1, max_nodes=16)
    st = _states_by_free(probe, per_f, seed=board[0] * 43 + board[1], f_max=18)
    probe.close()
    n = st.shape[0]
    eng = engine.Engine(board, n_games=n, max_nodes=16)
    eng.reset_roots(st)
    roots = eng.root_states()
    dev = eng.device
    E = eng.L * (eng.C + 1) + eng.C * (eng.L + 1)
    n_moves = E + 4  # room for every playout from a move index < 4
    gen = torch.Generator(device=dev)
    gen.manual_seed(17)
    eg16 = endgame.EndgameSolver(eng, 16)
    f = eg16.free_edges(roots)
    rollout = torch.arange(n, device=dev) >= n // 2  # _states_by_free: random masks first, then positions of real games
    table = solver.Solver(eng).solve() if board == (3, 3) else None
    g = solver_ref.Geometry(*board)
    roots_np = eng.states_to_numpy(roots)
    tree = torch.arange(n, device=dev)
    for mf in (0, 10, 12, 16):
        eg = endgame.EndgameSolver(eng, mf)
        want_margin = eg.margin(roots)
        for first in (0, 1):
            for kind in KINDS:
                B = _Buffers(eng, n_moves, gen)
                t, t0 = B.t, B.t0
                margin = torch.full((n,), 99, dtype=torch.int8, device=dev)
                eg.play_out(B.bufs, margin, kind, first=bool(first))
                torch.cuda.synchronize()
                hit = ((t0["moves"] >= 0) | bool(first)) & (t0["searching"] == 1) & (f <= mf)
                assert bool(hit.any()) or mf == 0
                # ---- replay every playout
                S = roots.clone()
                mi0 = t0["move_idx"]
                plies = torch.zeros((n,), dtype=torch.int64, device=dev)
                written = torch.zeros((n_moves, n), dtype=torch.bool, device=dev)
                for j in range(17):
                    live = hit & (eng.result(S) == 2) & eng.valid_moves(S).any(1) & (mi0 + j < n_moves)
                    if not bool(live.any()):
                        break
                    tl, rl = tree[live], (mi0 + j)[live]
                    Sl = S[live].contiguous()
                    assert torch.equal(t["h_states"][rl, tl], _published(eng, Sl)), (mf, first, kind, j)
                    opt = eg16.optimal_moves(Sl, kind)
                    assert bool(opt.any(1).all())
                    assert torch.equal(t["h_visits"][rl, tl], opt.int()), (mf, first, kind, j)
                    mv = t["h_moves"][rl, tl]
                    assert torch.equal(mv.long(), _draw(opt, t["uniforms"][rl, tl])), (mf, first, kind, j)
                    assert bool((t["h_stats"][rl, tl] == 0).all()) and bool((t["h_q"][rl, tl] == 0).all())
                    assert bool((t["h_active"][rl, tl] == 1).all())
                    written[rl, tl] = True
                    plies += live.long()
                    full_mv = torch.full((n,), -1, dtype=torch.int32, device=dev)
                    full_mv[live] = mv
                    eng.play(S, full_mv)
                ended = hit & (plies > 0)
                # every playout ran to a state with a result (a random mask with inconsistent scores may run out of edges)
                assert bool(((eng.result(S) != 2) | ~eng.valid_moves(S).any(1))[ended].all())
                assert bool((eng.result(S)[ended & rollout] != 2).all())
                # ---- the tree's outputs
                assert torch.equal(margin[hit], want_margin[hit]) and bool((margin[~hit] == 99).all()), (mf, first, kind)
                assert torch.equal(t["searching"], torch.where(hit, torch.zeros_like(t0["searching"]), t0["searching"]))
                assert torch.equal(t["reads"], torch.where(hit, torch.full_like(t0["reads"], -3), t0["reads"]))
                assert torch.equal(t["move_idx"], torch.where(ended, mi0 + plies - 1, mi0))
                assert int(t["left"]) == 100000 - int(hit.sum())
                for k in ("moves", "inv_temp", "uniforms", "reads_by_k", "noise_buf"):
                    assert torch.equal(t[k], t0[k]), k
                for k in ("h_states", "h_visits", "h_active", "h_moves", "h_stats", "h_q"):
                    assert torch.equal(t[k][~written], t0[k][~written]), k
                # ---- the played-out result has the sign of the exact margin (positions of real games: consistent scores)
                chk = ended & rollout
                if bool(chk.any()):
                    res = eng.result(S).long()
                    just = S.view(torch.uint8).reshape(n, 32)[:, 21].long()
                    tp = roots.view(torch.uint8).reshape(n, 32)[:, 20].long()
                    got = torch.where(just == tp, res, -res)
                    assert torch.equal(got[chk], torch.sign(margin[chk].long())), (mf, first, kind)
                if table is not None:
                    assert torch.equal(margin[hit], table.margin(roots[hit].contiguous()))
                elif mf in (12, 16) and kind == "outcome":
                    for r in torch.nonzero(hit).reshape(-1)[:16].tolist():
                        edges = int(roots_np["edges"][r][0]) | (int(roots_np["edges"][r][1]) << 64)
                        btc2 = (int(roots_np["btc2"][r][0]), int(roots_np["btc2"][r][1]))
                        assert int(margin[r]) == endgame_ref.endgame_moves(g, edges, btc2, int(roots_np["to_play"][r]))[1]
    if board == (1, 31):
        assert bool((f <= 16).any()) and bool((roots[:, 1] != 0).any())  # the second edge word was in play
    eng.close()


def test_error_paths(mods):
    engine, _, endgame, self_play, _ = mods
    eng = engine.Engine((3, 3), n_games=4, max_nodes=16)
    gen = torch.Generator(device=eng.device)
    gen.manual_seed(3)
    B = _Buffers(eng, 32, gen)
    z8 = torch.full((4,), -128, dtype=torch.int8, device=eng.device)
    for mf in (17, -1):
        with pytest.raises(engine.EngineError, match=r"dbaz_selfplay_exact_endgame: max_free must be in \[0, 16\], got %d" % mf):
            endgame.EndgameSolver(eng, mf).play_out(B.bufs, z8)
    with pytest.raises(engine.EngineError, match="dbaz_selfplay_exact_endgame: null exact_margin"):
        endgame.EndgameSolver(eng, 8).play_out(B.bufs, None)
    for kind in (2, -1):
        rc = eng.lib.dbaz_selfplay_exact_endgame(eng._h, ctypes.byref(B.bufs), ctypes.c_void_p(z8.data_ptr()), 8, kind, 0, eng._stream())
        assert rc != 0
        assert "dbaz_selfplay_exact_endgame: kind must be 0 (outcome) or 1 (margin)" in eng.lib.dbaz_last_error(eng._h).decode()
    with pytest.raises(ValueError, match="kind"):
        endgame.EndgameSolver(eng, 8).play_out(B.bufs, z8, kind="best")
    # the engine is still usable: a valid call runs
    endgame.EndgameSolver(eng, 8).play_out(B.bufs, z8, "margin", first=True)
    torch.cuda.synchronize()
    with pytest.raises(ValueError, match="DeepEndgameSolver"):
        endgame.DeepEndgameSolver(eng, 20).play_out(B.bufs, z8)
    for bad in (17, -1):
        with pytest.raises(ValueError, match="exact_endgame"):
            self_play.BatchedSelfPlay(eng, engine.FakeNetEvaluator(0), _params(), exact_endgame=bad)
    with pytest.raises(ValueError, match="exclude each other"):
        self_play.BatchedSelfPlay(eng, engine.FakeNetEvaluator(0), _params(), adjudicate=8, exact_endgame=8)
    p = _params()
    p.self_play.adjudicate = 6
    with pytest.raises(ValueError, match="exclude each other"):
        self_play.BatchedSelfPlay(eng, engine.FakeNetEvaluator(0), p, exact_endgame=10)
    with pytest.raises(ValueError, match="exact_policy"):
        self_play.BatchedSelfPlay(eng, engine.FakeNetEvaluator(0), _params(), exact_endgame=8, exact_policy="best")
    p = _params()
    p.self_play.exact_endgame = 6
    assert self_play.BatchedSelfPlay(eng, engine.FakeNetEvaluator(0), p).exact.max_free == 6
    assert self_play.BatchedSelfPlay(eng, engine.FakeNetEvaluator(0), _params()).exact is None
    eng.close()


def _device_rows(bsp):
    """per game slot: [(move index, state, visits, move, stats, q) of every recorded row], from the device history"""
    h = bsp._device_hist
    act = torch.stack(h["active"]).cpu().numpy()
    cols = [torch.stack(h[k]).cpu().numpy() for k in ("states", "visits", "moves", "stats", "q")]
    return [[(m,) + tuple(c[m, g] for c in cols) for m in range(act.shape[0]) if act[m, g]] for g in range(act.shape[1])]


def _same_row(a, b):
    return all(np.array_equal(np.asarray(x), np.asarray(y)) for x, y in zip(a, b))


def _z_by_game(bsp):
    bsp.rows, bsp.played_games = [], []
    bsp._rows_from_device(False)
    out = {}
    for r in bsp.rows:
        out.setdefault(r["game_idx"], []).append((r["player"], r["z"]))
    return out


def _check_exact_tail(eng, eg, kind, mf, S, vis, moves, stats, q, u=None, players=True):
    """rows S[0..] (int64 [k, 4] on the device) of one game from its first exact root on: positions with f <= mf and
    a result of NONE, visits = the optimal moves, zero statistics, moves that are optimal (and the replayed draw with u),
    each row the position the previous move leads to; returns the state after the last move"""
    assert bool((eg.free_edges(S) <= mf).all()) and bool((eng.result(S) == 2).all())
    opt = eg.optimal_moves(S, kind)
    assert torch.equal(torch.from_numpy(np.stack(vis)).to(eng.device), opt.int())
    assert np.all(np.stack(stats) == 0) and np.all(np.asarray(q) == 0)
    mv = torch.tensor(np.asarray(moves, dtype=np.int64), device=eng.device)
    assert bool(opt.gather(1, mv.unsqueeze(1)).all())
    if u is not None:
        assert torch.equal(mv, _draw(opt, u))
    nxt = S.clone()
    eng.play(nxt, mv.int())
    if players:
        assert torch.equal(_b22(nxt[:-1]), _b22(S[1:]))
    else:  # states rebuilt from feature planes name the player to move 0
        assert torch.equal(nxt[:-1, :2], S[1:, :2])
    assert int(eng.result(nxt[-1:])[0]) != 2  # the game ends at the first state with a result
    return nxt[-1:]


def _check_device_paths(eng, eg, off, on, mf, kind, path):
    """`on` (exact_endgame = mf) is `off` up to its first row with f <= mf, then exact rows to the end, with exact z"""
    g_off, g_on = _device_rows(off), _device_rows(on)
    z_off, z_on = _z_by_game(off), _z_by_game(on)
    h = on._device_hist
    final = h["final"]
    em = h["exact_margin"].cpu().numpy() if path == "async" else None
    n_ex, n_rows = 0, 0
    for g in range(eng.n_games):
        states = np.stack([r[1] for r in g_off[g]]) if g_off[g] else np.zeros((0, 4), np.int64)
        f = eg.free_edges(torch.from_numpy(states).to(eng.device).contiguous()).cpu().numpy() if len(states) else np.zeros(0)
        cut = int(np.argmax(f <= mf)) if (f <= mf).any() else None
        if cut is None:
            if em is not None:
                assert em[g] == -128
            assert len(g_on[g]) == len(g_off[g]) and all(_same_row(a, b) for a, b in zip(g_on[g], g_off[g])), g
            assert z_on.get(g) == z_off.get(g), g
            continue
        n_ex += 1
        assert len(g_on[g]) > cut and all(_same_row(a, b) for a, b in zip(g_on[g][:cut], g_off[g][:cut])), (g, cut)
        tail = g_on[g][cut:]
        n_rows += len(tail)
        assert [r[0] for r in tail] == list(range(tail[0][0], tail[0][0] + len(tail)))
        S = torch.from_numpy(np.stack([r[1] for r in tail])).to(eng.device).contiguous()
        assert torch.equal(S[0], torch.from_numpy(states[cut]).to(eng.device))  # the first exact root is the searched game's
        u = None
        if path == "async":
            u = h["uniforms"][torch.tensor([r[0] for r in tail], device=eng.device), g]
        end = _check_exact_tail(eng, eg, kind, mf, S, [r[2] for r in tail], [r[3] for r in tail], [r[4] for r in tail],
                                [r[5] for r in tail], u)
        root = S[:1]
        o = int(eg.outcome(root)[0])
        if path == "async":  # the tree keeps the exact root
            assert torch.equal(_b22(final[g:g + 1]), _b22(root)) and em[g] == int(eg.margin(root)[0])
        else:                # the game was played to its end on the tree
            assert torch.equal(_b22(final[g:g + 1]), _b22(end))
        tp = int(eng.states_to_numpy(root)["to_play"][0])
        assert [z for _, z in z_on[g]] == [o if p == tp else -o for p, _ in z_on[g]], g
        # the played-out result is the root's exact outcome
        res = int(eng.result(end)[0])
        just = int(eng.states_to_numpy(end)["just_played"][0])
        assert (res if just == tp else -res) == o, g
    return n_ex, n_rows


@pytest.mark.parametrize("path", ["async", "device"])
@pytest.mark.parametrize("board,n,mf", [((3, 3), 256, 12), ((3, 3), 256, 0), ((5, 5), 128, 10)])
@pytest.mark.parametrize("kind", ["fake", "endgame"])
def test_prefix_identity_device_paths(mods, board, n, mf, kind, path):
    engine, _, endgame, self_play, _ = mods
    eng = engine.Engine(board, n_games=n, max_nodes=1024, eval_cache=14)
    ev = _evaluator(engine, endgame, eng, kind)
    eg = endgame.EndgameSolver(eng, 16)
    policy = "margin" if board == (5, 5) else "outcome"
    runs = []
    for ex in (None, mf):
        bsp = self_play.BatchedSelfPlay(eng, ev, _params(), graph_waves=4, pending=1, adaptive=True, exact_endgame=ex,
                                        exact_policy=policy)
        fn = bsp.play_games_async if path == "async" else bsp.play_games_device
        info = fn(list(range(n)), seed=5)
        runs.append((bsp, info))
    (off, info_off), (on, info_on) = runs
    n_ex, n_rows = _check_device_paths(eng, eg, off, on, mf, policy, path)
    assert info_on["exact_games"] == n_ex and info_on["exact_rows"] == n_rows and info_on["adjudicated"] == 0
    assert info_off["exact_games"] == 0 and info_off["exact_rows"] == 0
    if mf == 0:
        assert n_ex == 0 and info_on["sims"] == info_off["sims"]
        for k in ("states", "visits", "active", "moves", "stats", "q"):
            assert all(torch.equal(a, b) for a, b in zip(off._device_hist[k], on._device_hist[k])), k
        for a, b in zip(off.device_samples(), on.device_samples()):
            assert torch.equal(a, b)
    else:
        assert n_ex > 0 and info_on["sims"] < info_off["sims"]
        if board == (5, 5):
            assert n_ex < n  # some games end at a majority first
        planes, pi, z, slot, mi = on.device_samples()
        assert planes.shape[0] == sum(len(r) for r in _device_rows(on))
    eng.close()


@pytest.mark.parametrize("board,n,mf", [((3, 3), 48, 12), ((3, 3), 48, 0), ((5, 5), 24, 10)])
@pytest.mark.parametrize("kind", ["fake", "endgame"])
def test_prefix_identity_host_rng(mods, board, n, mf, kind):
    """play_games (one legacy NumPy stream per game): every game with exact play is the same game without it up to its
    first root with f <= mf; from there its rows are exact, its moves are the draws rng.choice(A, 1, p=opt/k) of the
    same stream (no Dirichlet draw), and its z is the exact outcome of that root."""
    engine, _, endgame, self_play, _ = mods
    eng = engine.Engine(board, n_games=n, max_nodes=1024, eval_cache=14)
    ev = _evaluator(engine, endgame, eng, kind)
    eg = endgame.EndgameSolver(eng, 16)
    A = eng.A
    p = _params()
    alpha = p.self_play.noise[0]
    temp_sched = p.self_play.mcts.temperature
    seeds = [1000 + i for i in range(n)]
    runs = []
    for ex in (None, mf):
        bsp = self_play.BatchedSelfPlay(eng, ev, _params(), graph_waves=4, pending=1, adaptive=True, exact_endgame=ex)
        bsp.play_games(list(range(n)), seeds=seeds)
        runs.append((bsp, eng.root_states()))
    (off, _), (on, final_on) = runs
    rows_of = lambda b: {gi: [r for r in b.rows if r["game_idx"] == gi] for gi in range(n)}
    h_off, h_on = rows_of(off), rows_of(on)
    key = lambda r: (r["move_idx"], r["move"], r["player"], r["visits"], r["stats"], r["features"])
    n_ex = 0
    for gi in range(n):
        rows = h_off[gi]
        planes = np.stack([r["features"] for r in rows])
        f = eg.free_edges(eg.states_from_planes(torch.from_numpy(planes).to(eng.device))).cpu().numpy()
        if not (f <= mf).any():
            assert len(h_on[gi]) == len(rows) and all(_same_row(key(a), key(b)) for a, b in zip(h_on[gi], rows))
            assert [r["z"] for r in h_on[gi]] == [r["z"] for r in rows]
            assert on.played_games[gi][1] == off.played_games[gi][1] and on.played_games[gi][3] == off.played_games[gi][3]
            continue
        n_ex += 1
        cut = int(np.argmax(f <= mf))
        got = h_on[gi]
        assert len(got) > cut and all(_same_row(key(a), key(b)) for a, b in zip(got[:cut], rows[:cut])), (gi, cut)
        tail = got[cut:]
        S = eg.states_from_planes(torch.from_numpy(np.stack([r["features"] for r in tail])).to(eng.device)).contiguous()
        moves = on.played_games[gi][1]
        assert len(moves) == len(got)
        end = _check_exact_tail(eng, eg, "outcome", mf, S, [r["visits"] for r in tail], moves[cut:],
                                [np.asarray(r["stats"][:3]) for r in tail], [r["stats"][3] for r in tail], players=False)
        assert torch.equal(final_on[gi:gi + 1, :2], end[:, :2]) and int(eng.result(final_on[gi:gi + 1])[0]) != 2
        o = int(eg.outcome(S[:1])[0])
        tp = tail[0]["player"]
        assert [r["z"] for r in got] == [o if r["player"] == tp else -o for r in got]
        assert abs(on.played_games[gi][3]) == abs(o)
        # the game's own stream: the searched plies' Dirichlet and choice draws, then choice over the optimal moves
        rng = np.random.RandomState(seeds[gi])
        temp = None
        for j, r in enumerate(got):
            if j in temp_sched:
                temp = temp_sched[j]
            if j < cut:
                if alpha > 0:
                    rng.dirichlet(np.ones(A) * alpha, 1)
                rng.choice(A, 1, p=self_play._apply_temperature(r["visits"], temp))
            else:
                v = r["visits"]
                assert rng.choice(A, 1, p=v / v.sum())[0] == moves[j], (gi, j)
    assert (n_ex > 0) == (mf > 0)
    if mf == 0:
        assert off.get_datasets(0).equals(on.get_datasets(0))
    eng.close()


@pytest.mark.parametrize("share", [1.0, 0.5])
def test_solvable_start_states(mods, share):
    """Start states already solvable: played out exactly from the start, every row of those games exact; the loop ends
    (left == 0) on the asynchronous path; a mix of solvable and unsolvable start states on all three paths."""
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
                                        exact_endgame=mf)
        if path == "host":
            bsp.play_games(list(range(n)), seeds=list(range(n)), start_states=start.clone())
            info = None  # play_games returns the games, not the figures
            slot = np.asarray([r["game_idx"] for r in bsp.rows], dtype=np.int64)
            stats = np.asarray([r["stats"][:3] for r in bsp.rows])
            for gi in np.flatnonzero(solv):  # z of every row: the exact outcome of the start state, by player
                pz = [(r["player"], r["z"]) for r in bsp.rows if r["game_idx"] == gi]
                o = int(np.sign(want[gi]))
                assert [z for _, z in pz] == [o if pl == pz[0][0] else -o for pl, _ in pz], gi
        else:
            info = getattr(bsp, "play_games_" + path)(list(range(n)), seed=1, start_states=start.clone())
            if path == "async":
                em = bsp._device_hist["exact_margin"].cpu().numpy()
                assert np.array_equal(em[solv], want[solv])
            _, _, _, s_, _ = bsp.device_samples()
            slot = s_.cpu().numpy()
            stats = torch.stack(bsp._device_hist["stats"])[torch.stack(bsp._device_hist["active"])][:, 1:4].cpu().numpy()
            assert info["exact_games"] >= int(solv.sum()), path
            if share == 1.0:
                assert info["sims"] == 0 and info["exact_rows"] == len(slot) > 0, path
        mine = np.isin(slot, np.flatnonzero(solv))
        assert mine.sum() > 0 and np.all(stats[mine] == 0), path  # every row of those games is exact
        if share == 1.0:
            assert mine.all(), path
    eng.close()


def test_padded_chunk_frames_and_grading(mods):
    """play_shard with a short last chunk (padding games of index -1) keeps exact rows; batch_from_selfplay, get_datasets()
    and played_games agree row for row; grade_samples on EndgameSolver(max_free) grades every exact row as optimal."""
    engine, solver, endgame, self_play, _ = mods
    from dotsboxesaz_b200 import samples
    n, mf = 64, 12
    eng = engine.Engine((3, 3), n_games=n, max_nodes=1024, eval_cache=14)
    p = _params()
    p.self_play.exact_endgame = mf
    p.self_play.mcts.max_async_searches = 1
    batch, frames, info = self_play.play_shard(p, 0, eng, engine.FakeNetEvaluator(0), list(range(40)), want_frames=True)
    eg = endgame.EndgameSolver(eng, 16)
    f = eg.free_edges(eg.states_from_planes(batch.planes))
    assert len(batch) > 0 and bool((f <= mf).any()) and bool((f > mf).any())
    df = frames[0]
    assert len(df) == len(batch) and set(df.index.get_level_values("game_idx")) <= set(range(40))
    meta = batch.meta.cpu().numpy()
    order = np.lexsort((meta[:, 2], meta[:, 1]))
    assert np.array_equal(df["z"].to_numpy().astype(np.float32), batch.z.cpu().numpy()[order])
    assert np.array_equal(df[[c for c in df.columns if c.startswith("pi_")]].to_numpy().astype(np.float32), batch.pi.cpu().numpy()[order])
    # one more chunk by hand: played_games, the DataFrame and the sample batch
    bsp = self_play.BatchedSelfPlay(eng, engine.FakeNetEvaluator(0), p)
    idx = list(range(40)) + [-1] * 24
    info = bsp.play_games_async(idx, seed=9)
    assert info["exact_games"] > 0 and info["exact_rows"] > 0
    b = samples.batch_from_selfplay(bsp, 0)
    planes, pi, z, slot, mi = bsp.device_samples()
    real = torch.as_tensor(np.asarray(idx), device=slot.device)[slot] >= 0
    assert len(b) == int(real.sum()) and torch.equal(b.z, z[real].float()) and torch.equal(b.pi, pi[real].float())
    df = bsp.get_datasets(0, False)
    df = df[df.index.get_level_values("game_idx") >= 0]
    m = b.meta.cpu().numpy()
    order = np.lexsort((m[:, 2], m[:, 1]))
    assert np.array_equal(df["z"].to_numpy().astype(np.float32), b.z.cpu().numpy()[order])
    ex_rows = df[(df["tree_size"] == 0) & (df["max_deepness"] == 0)]
    assert len(ex_rows) > 0 and bool((ex_rows["q_value"] == 0).all())
    bsp._rows_from_device(False)
    rz = np.asarray([r["z"] for r in bsp.rows if r["game_idx"] >= 0], dtype=np.float32)
    assert np.array_equal(rz, df["z"].to_numpy().astype(np.float32))
    for gi, mv, vis, zg in bsp.played_games:
        if gi >= 0:
            zs = df.xs(gi, level="game_idx")["z"].to_numpy()
            assert len(vis) == len(zs) == len(mv) and set(np.abs(zs)) <= {abs(zg)}
    # grading: the exact rows are exactly the rows EndgameSolver(mf) solves, all optimal, z all agreeing
    gr = solver.grade_samples(endgame.EndgameSolver(eng, mf), b)
    n_exact = int((eg.free_edges(eg.states_from_planes(b.planes)) <= mf).sum())
    assert gr["n_solved"] == n_exact == len(ex_rows) > 0
    assert gr["optimal_move_rate"] == 1.0 and gr["optimal_mass"] == pytest.approx(1.0, abs=1e-6) and gr["z_agreement"] == 1.0
    eng.close()


def test_coach_generation(mods, tmp_path):
    """One learn_to_play generation on 3x3 with exact_endgame on: rows with f <= max_free are exported, with the exact
    rows' zero tree statistics."""
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
    params.self_play.exact_endgame = 12
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
    assert (f <= 12).any() and (f > 12).any()
    ex = data[f <= 12]
    assert (ex["tree_size"] == 0).all() and (ex["max_deepness"] == 0).all() and (ex["q_value"] == 0).all()
    eng.close()
