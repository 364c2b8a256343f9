"""GPU: the exact endgame solver (csrc/dbaz_endgame.cuh, dotsboxesaz_b200/endgame.py).  Byte for byte against the
32-edge table on every board that has one, for every number of free edges 0 .. 16 and max_free 0 / 7 / 10 / 16 (both
tiers and their boundary); against the NumPy sub-table on boards up to 7x7 (two edge words, actions >= 64); the
evaluator against SolverEvaluator and the inner evaluator, bit for bit, and inside every search mode; grading of 5x5
self-play against a host recount; the error paths."""
import copy

import numpy as np
import pytest

import endgame_ref

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def mods():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from dotsboxesaz_b200 import endgame, engine, solver
    from oracle import solver_ref
    return engine, solver, endgame, solver_ref


SMALL = [(1, 1), (1, 2), (1, 3), (1, 4), (1, 5), (1, 6), (1, 7), (2, 1), (3, 1), (4, 1), (5, 1), (6, 1), (7, 1), (2, 2), (2, 3), (3, 2),
         (2, 4), (4, 2), (3, 3)]
MAX_FREE = (0, 7, 10, 16)


def _real_actions(L, C):
    cols, plane = C + 1, (L + 1) * (C + 1)
    return [a for a in range(2 * plane) if (a < plane and a % cols < C) or (a >= plane and (a - plane) // cols < L)]


def _words(bits):
    """edge words int64 [n, 2] of action bits [n, 128]"""
    sh = torch.arange(64, device=bits.device)
    return torch.stack([(bits[:, :64].long() << sh).sum(1), (bits[:, 64:].long() << sh).sum(1)], 1)


def _mask_states(eng, n_free, n, gen):
    """n states with exactly n_free free real edges at random, random scores and player to move"""
    dev = eng.device
    real = torch.tensor(_real_actions(eng.L, eng.C), dtype=torch.int64, device=dev)
    E = real.numel()
    ranks = torch.rand((n, E), generator=gen, device=dev).argsort(1)
    bits = torch.zeros((n, 128), dtype=torch.int64, device=dev)
    bits[:, real] = (ranks >= n_free).long()
    st = eng.new_states(1).repeat(n, 1)
    st[:, :2] = _words(bits)
    v16 = st.view(torch.int16)
    LC = eng.L * eng.C
    v16[:, 8] = torch.randint(-LC, LC + 1, (n,), generator=gen, device=dev).to(torch.int16)
    v16[:, 9] = torch.randint(-LC, LC + 1, (n,), generator=gen, device=dev).to(torch.int16)
    v16[:, 10] = (v16[:, 10] & ~0xff) | torch.randint(0, 2, (n,), generator=gen, device=dev).to(torch.int16)
    return st.contiguous()


def _rollout_states(eng, depth, gen):
    """states after depth[i] uniform random legal moves (the game goes on past a majority)"""
    n = depth.shape[0]
    st = eng.new_states(n)
    for ply in range(int(depth.max()) if n else 0):
        valid = eng.valid_moves(st).double()
        live = (depth > ply) & (valid.sum(1) > 0)
        mv = torch.multinomial(valid + (valid.sum(1, keepdim=True) == 0).double(), 1, generator=gen).reshape(-1)
        eng.play(st, torch.where(live, mv, torch.full_like(mv, -1)).int())
    return st


def _states_by_free(eng, per_f, seed, f_max=16):
    """per_f random-mask states and per_f rollout states stopped at E - f plies, for every f in 0 .. min(E, f_max)"""
    gen = torch.Generator(device=eng.device)
    gen.manual_seed(seed)
    E = len(_real_actions(eng.L, eng.C))
    fs = range(min(E, f_max) + 1)
    masks = torch.cat([_mask_states(eng, f, per_f, gen) for f in fs])
    depth = torch.cat([torch.full((per_f,), E - f, dtype=torch.int64, device=eng.device) for f in fs])
    return torch.cat([masks, _rollout_states(eng, depth, gen)]).contiguous()


def _solved(engine, solver, board, n_games=1, **kw):
    eng = engine.Engine(board, n_games=n_games, max_nodes=kw.pop("max_nodes", 16), **kw)
    return eng, solver.Solver(eng).solve()


@pytest.mark.parametrize("board", SMALL + [(3, 4), (2, 6)])
def test_moves_equal_32_edge_table(mods, board):
    """>= 2000 states for every f (random masks and rollouts): rows with f <= max_free equal Solver.moves byte for byte,
    every other row is all -128."""
    engine, solver, endgame, _ = mods
    eng, s = _solved(engine, solver, board)
    st = _states_by_free(eng, 1000, seed=board[0] * 31 + board[1])
    mm, mg = s.moves(st)
    f = endgame.EndgameSolver(eng).free_edges(st)
    assert int(f.bincount().min()) >= 2000
    for mf in MAX_FREE:
        eg = endgame.EndgameSolver(eng, mf)
        emm, emg = eg.moves(st)
        ok = f <= mf
        assert torch.equal(eg.solvable(st), ok)
        assert torch.equal(emm[ok], mm[ok]) and torch.equal(emg[ok], mg[ok]), (board, mf)
        assert bool((emm[~ok] == -128).all()) and bool((emg[~ok] == -128).all()), (board, mf)
        assert torch.equal(eg.outcome(st)[ok], torch.sign(mg[ok])) and bool((eg.outcome(st)[~ok] == -128).all())
        assert torch.equal(eg.optimal_moves(st, "margin")[ok], s.optimal_moves(st, "margin")[ok])
    del s
    eng.close()
    torch.cuda.empty_cache()


def test_many_passes_3x3(mods):
    """300 000 rows: more than one pass of the persistent grid over the rows, both tiers mixed in every pass."""
    engine, solver, endgame, _ = mods
    eng, s = _solved(engine, solver, (3, 3))
    gen = torch.Generator(device=eng.device)
    gen.manual_seed(9)
    st = torch.cat([_mask_states(eng, f, 300_000 // 17 + 1, gen) for f in range(17)])
    st = st[torch.randperm(st.shape[0], generator=gen, device=eng.device)].contiguous()
    mm, mg = s.moves(st)
    for mf in (16, 12):
        eg = endgame.EndgameSolver(eng, mf)
        emm, emg = eg.moves(st)
        ok = eg.solvable(st)
        assert torch.equal(emm[ok], mm[ok]) and torch.equal(emg[ok], mg[ok])
        assert bool((emm[~ok] == -128).all()) and bool((emg[~ok] == -128).all())
    eng.close()


LARGE = [(4, 4), (5, 5), (6, 6), (7, 7), (4, 7), (1, 31), (31, 1)]


def _host_rows(eng, st):
    rec = eng.states_to_numpy(st)
    return [(int(r["edges"][0]) | (int(r["edges"][1]) << 64), (int(r["btc2"][0]), int(r["btc2"][1])), int(r["to_play"])) for r in rec]


@pytest.mark.parametrize("board", LARGE)
def test_large_boards_equal_numpy(mods, board):
    """Move margins, final margins and both evaluator modes against endgame_numpy, f = 0 .. 16."""
    engine, _, endgame, solver_ref = mods
    eng = engine.Engine(board, n_games=1, max_nodes=16)
    st = _states_by_free(eng, 6, seed=board[0] * 37 + board[1])
    eg = endgame.EndgameSolver(eng, 16)
    mm, mg = (x.cpu().numpy() for x in eg.moves(st))
    n, A = st.shape[0], eng.A
    P = torch.full((n, A), 7.0, device=eng.device)
    V = torch.full((n,), 7.0, device=eng.device)
    eg.evaluate(eng, st, P, V, 0)
    V1 = V.clone()
    eg.evaluate(eng, st, P, V1, 1)
    P, V, V1 = P.cpu().numpy(), V.cpu().numpy(), V1.cpu().numpy()
    g = solver_ref.Geometry(*board)
    high = 0
    for r, (edges, btc2, tp) in enumerate(_host_rows(eng, st)):
        want_mm, want_final = endgame_ref.endgame_moves(g, edges, btc2, tp)
        assert np.array_equal(mm[r].astype(np.int64), want_mm), (board, r)
        assert int(mg[r]) == want_final
        o = int(np.sign(want_final))
        opt = (want_mm != -128) & (np.sign(want_mm) == o)
        k = int(opt.sum())
        assert np.array_equal(P[r], np.where(opt, np.float32(1.0) / np.float32(k) if k else 0.0, 0.0).astype(np.float32))
        assert V[r] == o and V1[r] == np.float32(want_final) / np.float32(g.LC)
        high += int((want_mm[64:] != -128).any())
    assert high > 0 or g.A <= 64  # actions >= 64 were graded
    eng.close()


def _fake(eng, st, kind=0):
    n = st.shape[0]
    P = torch.full((n, eng.A), 7.0, device=eng.device)
    V = torch.full((n,), 7.0, device=eng.device)
    eng.fake_nn(st, kind, P, V)
    return P, V


def _bits(x):
    return x.contiguous().view(torch.int32)


def test_evaluator_rows_against_solver_evaluator(mods):
    """3x3: on rows with f <= max_free the endgame evaluator's output is SolverEvaluator's, bit for bit; every other row is
    the inner evaluator's; priors="inner" keeps the inner priors everywhere."""
    engine, solver, endgame, _ = mods
    eng, s = _solved(engine, solver, (3, 3))
    gen = torch.Generator(device=eng.device)
    gen.manual_seed(3)
    E = 24
    st = _rollout_states(eng, torch.randint(0, E + 1, (6000,), generator=gen, device=eng.device), gen)
    f = endgame.EndgameSolver(eng).free_edges(st)
    assert bool((f <= 16).any()) and bool((f > 16).any())
    for mode in (0, 1):
        Ps, Vs = _fake(eng, st)
        s.evaluate(eng, st, Ps, Vs, mode)
        for mf in MAX_FREE + (12,):
            eg = endgame.EndgameSolver(eng, mf)
            ok = f <= mf
            P0, V0 = _fake(eng, st)
            P, V = P0.clone(), V0.clone()
            eg.evaluate(eng, st, P, V, mode)
            assert torch.equal(_bits(P[ok]), _bits(Ps[ok])) and torch.equal(_bits(V[ok]), _bits(Vs[ok])), (mode, mf)
            assert torch.equal(_bits(P[~ok]), _bits(P0[~ok])) and torch.equal(_bits(V[~ok]), _bits(V0[~ok])), (mode, mf)
            P, V = P0.clone(), V0.clone()
            eg.evaluate(eng, st, P, V, mode, keep_priors=True)
            assert torch.equal(_bits(P), _bits(P0))
            assert torch.equal(_bits(V[ok]), _bits(Vs[ok])) and torch.equal(_bits(V[~ok]), _bits(V0[~ok]))
    eng.close()


def test_evaluator_wrapper(mods):
    engine, solver, endgame, _ = mods
    eng, s = _solved(engine, solver, (2, 2))
    eg = endgame.EndgameSolver(eng, 8)
    assert endgame.EndgameEvaluator(engine.FakeNetEvaluator(0), eg).engine_launches == 2
    assert endgame.EndgameEvaluator(solver.SolverEvaluator(s), eg, "margin", "inner").engine_launches == 2
    with pytest.raises(ValueError):
        endgame.EndgameEvaluator(engine.FakeNetEvaluator(0), eg, value="bogus")
    with pytest.raises(ValueError):
        endgame.EndgameEvaluator(engine.FakeNetEvaluator(0), eg, priors="bogus")
    other = engine.Engine((3, 3), n_games=4, max_nodes=64)
    with pytest.raises(ValueError):
        other.run_search(10, endgame.EndgameEvaluator(engine.FakeNetEvaluator(0), eg))
    other.close()
    eng.close()


def _snapshot(eng):
    vis = eng.root_visits().cpu().numpy()
    W, P, S, U = (x.cpu().numpy() for x in eng.root_children())
    st, rW, q = (x.cpu().numpy() for x in eng.tree_stats())
    return {"visits": vis, "W": W.view(np.uint32), "priors": P.view(np.uint64), "stats": st[:, :7], "root_W": rW.view(np.uint32)}


def _search_moves(eng, ev, roots, sims, moves, **kw):
    eng.reset_roots(roots)
    out = []
    for _ in range(moves):
        eng.run_search(sims, ev, **kw)
        snap = _snapshot(eng)
        out.append(snap)
        eng.advance_roots(np.where(snap["visits"].sum(1) > 0, snap["visits"].argmax(1), -1).astype(np.int32), reuse=True)
    return out


@pytest.mark.parametrize("loop", ["device_loop", "host_loop"])
@pytest.mark.parametrize("value,max_free", [("outcome", 12), ("margin", 8)])
def test_search_production_schedule_bit_exact(mods, value, max_free, loop):
    """2048 trees of 5x5 from roots 36 .. 44 plies deep: eval cache + compact rows + adaptive ladder (+ device-driven
    loop) == the plain wave loop, bit for bit; the endgame evaluator changes the search."""
    engine, _, endgame, _ = mods
    n, sims = 2048, 200
    plain = engine.Engine((5, 5), n_games=n, max_nodes=4 * sims + 64)
    ev = endgame.EndgameEvaluator(engine.FakeNetEvaluator(0), endgame.EndgameSolver(plain, max_free), value)
    gen = torch.Generator(device=plain.device)
    gen.manual_seed(7)
    roots = _rollout_states(plain, torch.randint(36, 45, (n,), generator=gen, device=plain.device), gen)
    roots = torch.where((plain.result(roots) == 2).unsqueeze(1), roots, plain.new_states(n))
    ref = _search_moves(plain, ev, roots, sims, 2)
    info_plain = plain.status()
    fake = _search_moves(plain, engine.FakeNetEvaluator(0), roots, sims, 1)
    assert not np.array_equal(fake[0]["visits"], ref[0]["visits"])
    eng = engine.Engine((5, 5), n_games=n, max_nodes=4 * sims + 64, eval_cache=16)
    eng.device_loop = loop == "device_loop"
    got = _search_moves(eng, ev, roots.clone(), sims, 2, graph_waves=4, adaptive=True)
    assert eng.device_loop == (loop == "device_loop")
    info = eng.status()
    for m, (a, b) in enumerate(zip(ref, got)):
        for key in a:
            assert np.array_equal(a[key], b[key]), (value, m, key)
    assert info["sims"] == info_plain["sims"] and info["cache_hits"] > 0
    eng.close()
    plain.close()


def _params(num_read=64, noise=(0.0, 0.0)):
    from dotsboxesaz_b200 import configuration
    p = copy.deepcopy(configuration.simple)
    p.self_play.mcts.mcts_num_read = num_read
    p.self_play.noise = noise
    return p


def test_selfplay_and_grade_samples_5x5(mods):
    """Self-play through play_games_async with the endgame evaluator from roots 30 plies deep; grade_samples with an
    EndgameSolver against a host recount from margin_minimax over the solvable rows."""
    engine, solver, endgame, solver_ref = mods
    from dotsboxesaz_b200 import samples, self_play
    n, max_free = 64, 12
    eng = engine.Engine((5, 5), n_games=n, max_nodes=1024, eval_cache=14)
    eg = endgame.EndgameSolver(eng, max_free)
    ev = endgame.EndgameEvaluator(engine.FakeNetEvaluator(0), eg)
    gen = torch.Generator(device=eng.device)
    gen.manual_seed(4)
    start = _rollout_states(eng, torch.full((n,), 30, dtype=torch.int64, device=eng.device), gen)
    start = torch.where((eng.result(start) == 2).unsqueeze(1), start, eng.new_states(n)).contiguous()
    bsp = self_play.BatchedSelfPlay(eng, ev, _params(64, (0.8, 0.25)), graph_waves=4, pending=1, adaptive=True)
    bsp.play_games_async(list(range(n)), seed=3, start_states=start)
    batch = samples.batch_from_selfplay(bsp, 0)
    got = solver.grade_samples(eg, batch)
    g = solver_ref.Geometry(5, 5)
    x = batch.planes.cpu().numpy().astype(np.int64)
    pi = batch.pi.cpu().numpy().astype(np.float64)
    z = batch.z.cpu().numpy().astype(np.float64)
    P = g.plane
    memo, rows = {}, []
    for r in range(len(batch)):
        edges = sum(1 << a for a in range(2 * P) if x[r, a])
        if len(endgame_ref.free_edges(g, edges)) > max_free:
            continue
        k = int(np.int8(np.uint8(x[r, 2 * P])))
        d = g.LC - k - g.closed_boxes(edges)
        o = np.sign(d + endgame_ref.margin_minimax(g, edges, memo))
        opt = np.zeros(eng.A, bool)
        for a in endgame_ref.free_edges(g, edges):
            e2 = edges | (1 << a)
            c = sum(1 for b in g.boxes_of[a] if e2 & g.box_mask[b] == g.box_mask[b])
            v = endgame_ref.margin_minimax(g, e2, memo)
            opt[a] = np.sign(d + (c + v if c else -v)) == o
        rows.append((opt[int(np.argmax(pi[r]))], float((pi[r] * opt).sum()), float(np.sign(z[r]) == o)))
    rows = np.array(rows, dtype=np.float64)
    assert got["n"] == len(batch) and got["n_solved"] == len(rows) > 0 and len(rows) < len(batch)
    assert got["optimal_move_rate"] == pytest.approx(rows[:, 0].mean(), abs=1e-12)
    assert got["optimal_mass"] == pytest.approx(rows[:, 1].mean(), abs=1e-12)
    assert got["z_agreement"] == pytest.approx(rows[:, 2].mean(), abs=1e-12)
    # the rebuilt states carry the sample's key
    st = eg.states_from_planes(batch.planes)
    assert torch.equal(eng.features(st, torch.int16).reshape(len(batch), -1).to(torch.uint8), batch.planes)
    eng.close()


@pytest.mark.parametrize("board", [(3, 3), (7, 7)])
def test_states_from_planes_both_words(mods, board):
    engine, _, endgame, _ = mods
    eng = engine.Engine(board, n_games=1, max_nodes=16)
    gen = torch.Generator(device=eng.device)
    gen.manual_seed(6)
    E = len(_real_actions(*board))
    st = _rollout_states(eng, torch.randint(0, E + 1, (512,), generator=gen, device=eng.device), gen)
    eg = endgame.EndgameSolver(eng)
    planes = eng.features(st, torch.int16).reshape(512, -1)
    back = eg.states_from_planes(planes)
    assert torch.equal(back[:, :2], st[:, :2])
    assert torch.equal(eng.features(back, torch.int16).reshape(512, -1), planes)
    assert torch.equal(eg.moves(back)[1], eg.moves(st)[1])
    eng.close()


def test_error_paths(mods):
    engine, _, endgame, _ = mods
    eng = engine.Engine((5, 5), n_games=1, max_nodes=16)
    st = eng.new_states(1)
    P = torch.zeros((1, eng.A), device=eng.device)
    V = torch.zeros((1,), device=eng.device)
    for mf in (17, -1):
        eg = endgame.EndgameSolver(eng, mf)
        with pytest.raises(engine.EngineError, match=r"dbaz_endgame_moves: max_free must be in \[0, 16\], got %d" % mf):
            eg.moves(st)
        with pytest.raises(engine.EngineError, match=r"dbaz_endgame_eval: max_free must be in \[0, 16\], got %d" % mf):
            eg.evaluate(eng, st, P, V)
    eg = endgame.EndgameSolver(eng, 16)
    with pytest.raises(engine.EngineError, match="mode must be 0"):
        eg.evaluate(eng, st, P, V, mode=2)
    with pytest.raises(engine.EngineError, match="dbaz_endgame_eval: null buffer"):
        eg.evaluate(eng, st, None, V)
    with pytest.raises(engine.EngineError, match="dbaz_endgame_eval: null buffer"):
        eg.evaluate(eng, st, P, None)
    buf = torch.zeros((1, eng.A), dtype=torch.int8, device=eng.device)
    for args in ((None, buf, buf), (st, None, buf), (st, buf, None)):
        assert eng.lib.dbaz_endgame_moves(eng._h, *(engine._ptr(a) for a in args), 16, 1, eng._stream()) != 0
        assert b"dbaz_endgame_moves: null buffer" in eng.lib.dbaz_last_error(eng._h)
    eng.close()
