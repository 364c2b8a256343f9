"""GPU: the exact solver (csrc/dbaz_solver.cuh, dotsboxesaz_b200/solver.py).  Full tables bit for bit against the NumPy
retrograde reference on every board with at most 24 edges; on 3x4, 4x3 and 2x6 the recurrence on sampled masks with
successors and closed boxes from the engine's own play kernel, symmetry and transposition invariance; per-state
queries against minimax and the engine's rules; perfect play against itself; the evaluator inside every search mode;
play_vs_solver and grade_samples against host recounts."""
import copy

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def mods():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from dotsboxesaz_b200 import engine, solver
    from oracle import solver_ref
    return engine, solver, solver_ref


_REF = {}


def _ref_table(solver_ref, board):
    if board not in _REF:
        _REF[board] = solver_ref.retrograde_numpy(*board)
    return _REF[board]


def _solved(engine, solver, board, n_games=1, **kw):
    eng = engine.Engine(board, n_games=n_games, max_nodes=kw.pop("max_nodes", 16), **kw)
    return eng, solver.Solver(eng).solve()


def _compact_to_edges(s, M):
    """action-space edge words (int64) of compact masks M (int64 tensor)"""
    act = torch.tensor(_real_actions(s.L, s.C), dtype=torch.int64, device=M.device)
    bits = (M.unsqueeze(1) >> torch.arange(s.E, device=M.device)) & 1
    return (bits << act).sum(1)


def _real_actions(L, C):
    cols, plane = C + 1, (L + 1) * (C + 1)
    return [a for a in range(2 * plane) if (a < plane and a % cols < C) or (a >= plane and (a - plane) // cols < L)]


def _states_of(eng, edges, btc2=(100, 100), to_play=0):
    """packed states with the given edge words (boxes-to-close large enough that no game is over)"""
    n = edges.shape[0]
    st = eng.new_states(1).repeat(n, 1)
    st[:, 0] = edges
    v16 = st.view(torch.int16)
    v16[:, 8] = btc2[0]
    v16[:, 9] = btc2[1]
    v16[:, 10] = (v16[:, 10] & ~0xff) | to_play
    return st.contiguous()


SMALL = [(1, 1), (1, 2), (1, 3), (1, 4), (1, 5), (1, 6), (1, 7), (2, 1), (3, 1), (4, 1), (5, 1), (6, 1), (7, 1), (2, 2), (2, 3), (3, 2),
         (2, 4), (4, 2), (3, 3)]


@pytest.mark.parametrize("board", SMALL)
def test_full_table_equals_numpy_retrograde(mods, board):
    engine, solver, solver_ref = mods
    eng, s = _solved(engine, solver, board)
    assert np.array_equal(s.table.cpu().numpy(), _ref_table(solver_ref, board))
    eng.close()


_LARGE = {}


def _large(mods, board):
    engine, solver, _ = mods
    if board not in _LARGE:  # 3x4, 4x3 (2 GiB each) and 2x6 (4 GiB) are solved once for the module
        _LARGE[board] = _solved(engine, solver, board)
    return _LARGE[board]


@pytest.mark.parametrize("board", [(3, 4), (4, 3), (2, 6)])
def test_large_board_recurrence_sampled(mods, board):
    """>= 10^6 masks over all layers: v(M) = max over free j of (c ? c + v(M|j) : -v(M|j)) with the successor state and c
    from dbaz_game_play, not from the solver's box masks; no sentinel anywhere."""
    eng, s = _large(mods, board)
    E, dev = s.E, eng.device
    T = s.table
    assert int((T == -128).sum()) == 0
    gen = torch.Generator(device=dev)
    gen.manual_seed(1)
    per_layer = -(-1_000_000 // E)
    act = torch.tensor(_real_actions(s.L, s.C), dtype=torch.int32, device=dev)
    checked = 0
    for k in range(E):
        ranks = torch.rand((per_layer, E), generator=gen, device=dev).argsort(1).argsort(1)
        M = ((ranks < k).long() << torch.arange(E, device=dev)).sum(1)
        edges = _compact_to_edges(s, M)
        best = torch.full((per_layer,), -1000, dtype=torch.int32, device=dev)
        for j in range(E):
            st = _states_of(eng, edges)
            ncl, _ = eng.play(st, act[j].repeat(per_layer))
            free = ((M >> j) & 1) == 0
            assert torch.equal(ncl >= 0, free)
            succ = st[:, 0]
            # successor mask back to compact form from the played state's edges
            bits = (succ.unsqueeze(1) >> act.long()) & 1
            Ms = (bits << torch.arange(E, device=dev)).sum(1)
            assert torch.equal(torch.where(free, Ms, M | (1 << j)), M | (1 << j))
            v = T[Ms].int()
            val = torch.where(ncl > 0, ncl + v, -v)
            best = torch.where(free, torch.maximum(best, val), best)
        assert torch.equal(best, T[M].int()), (board, k)
        checked += per_layer
    assert checked >= 1_000_000


def _permute_compact(s, M, perm):
    """compact masks of the positions whose edge a is edge perm[a] of M (dots_boxes_nn._edge_permutations)"""
    dev = M.device
    real = _real_actions(s.L, s.C)
    comp = {a: j for j, a in enumerate(real)}
    src = torch.tensor([comp[perm[a]] for a in real], dtype=torch.int64, device=dev)  # new compact j takes old compact src[j]
    bits = (M.unsqueeze(1) >> src) & 1
    return (bits << torch.arange(s.E, device=dev)).sum(1)


@pytest.mark.parametrize("board", [(3, 4), (4, 3), (2, 6)])
def test_large_board_symmetry_invariance(mods, board):
    from dotsboxesaz_b200.dots_boxes.dots_boxes_nn import _edge_permutations
    eng, s = _large(mods, board)
    gen = torch.Generator(device=eng.device)
    gen.manual_seed(2)
    M = torch.randint(0, 1 << s.E, (1 << 22,), generator=gen, device=eng.device, dtype=torch.int64)
    for perm in _edge_permutations(*board)[1:].tolist():
        assert torch.equal(s.table[M], s.table[_permute_compact(s, M, perm)])


def test_3x4_equals_4x3_transposed(mods):
    _, s34 = _large(mods, (3, 4))
    _, s43 = _large(mods, (4, 3))
    L, C = 3, 4
    cols, plane = C + 1, (L + 1) * (C + 1)
    cols_t = L + 1
    real, real_t = _real_actions(L, C), _real_actions(C, L)
    comp_t = {a: j for j, a in enumerate(real_t)}
    dst = []
    for a in real:  # edge of dots (y, x)-(y', x') -> edge of dots (x, y)-(x', y') on the transposed board
        p, rem = divmod(a, plane)
        l, c = divmod(rem, cols)
        dst.append(comp_t[plane + c * cols_t + l] if p == 0 else comp_t[c * cols_t + l])
    dev = s34.table.device
    for lo in range(0, 1 << 31, 1 << 26):  # the whole table
        M = torch.arange(lo, lo + (1 << 26), dtype=torch.int64, device=dev)
        Mt = torch.zeros_like(M)
        for j in range(31):
            Mt |= ((M >> j) & 1) << int(dst[j])
        assert torch.equal(s34.table[lo:lo + (1 << 26)], s43.table[Mt]), lo


def _random_states(eng, n, seed, max_depth=None):
    """n positions from uniform random games stopped after a random number of plies (terminal ones included)"""
    dev = eng.device
    gen = torch.Generator(device=dev)
    gen.manual_seed(seed)
    E = eng.L * (eng.C + 1) + eng.C * (eng.L + 1)
    depth = torch.randint(0, (max_depth or E) + 1, (n,), generator=gen, device=dev)
    st = eng.new_states(n)
    for ply in range(E):
        valid = eng.valid_moves(st).double()
        live = (depth > ply) & (eng.result(st) == 2) & (valid.sum(1) > 0)
        mv = torch.multinomial(valid + (valid.sum(1, keepdim=True) == 0).double(), 1, generator=gen).reshape(-1)
        eng.play(st, torch.where(live, mv, torch.full_like(mv, -1)).int())
    return st


def _host_state(eng, st):
    rec = eng.states_to_numpy(st)
    return [(int(r["edges"][0]), (int(r["btc2"][0]), int(r["btc2"][1])), int(r["to_play"])) for r in rec]


@pytest.mark.parametrize("board", [(2, 2), (2, 3), (3, 2), (3, 3), (3, 4)])
def test_states_from_random_rollouts(mods, board):
    engine, solver, solver_ref = mods
    n = 4096
    if board == (3, 4):
        eng, s = _large(mods, board)
    else:
        eng, s = _solved(engine, solver, board)
    st = _random_states(eng, n, seed=11)
    mm, mg = s.moves(st)
    res = eng.result(st)
    term = res != 2
    # terminal: the reference's result
    assert bool(term.any()) and bool((~term).any())
    assert torch.equal(torch.sign(mg)[term], res[term])
    # every non-terminal position has an outcome-optimal move
    opt = s.optimal_moves(st, "outcome")
    assert bool(opt[~term].any(1).all())
    assert torch.equal(s.outcome(st), torch.sign(mg)) and torch.equal(s.margin(st), mg) and torch.equal(s.move_margins(st), mm)
    # move margins recounted with the engine's play kernel and the table
    A = eng.A
    legal = eng.valid_moves(st)
    assert torch.equal(legal, mm != -128)
    rep = st.repeat_interleave(A, 0).contiguous()
    acts = torch.arange(A, device=eng.device, dtype=torch.int32).repeat(n)
    raw = st.view(torch.uint8).reshape(n, 32)
    tp = raw[:, 20].long()
    btc2 = raw[:, 16:20].contiguous().view(torch.int16).reshape(n, 2).long()
    ncl, _ = eng.play(rep, acts)
    real = torch.tensor(_real_actions(*board), dtype=torch.int64, device=eng.device)
    comp = lambda w: ((((w.unsqueeze(1) >> real) & 1)) << torch.arange(s.E, device=eng.device)).sum(1)
    M = comp(st[:, 0])
    Ms = comp(rep[:, 0]).reshape(n, A)
    d = (btc2.gather(1, (1 - tp).unsqueeze(1)) - btc2.gather(1, tp.unsqueeze(1))).squeeze(1) // 2
    v = s.table[Ms].int()
    c = ncl.reshape(n, A)
    want = torch.where(legal, d.unsqueeze(1) + torch.where(c > 0, c + v, -v), torch.full_like(v, -128))
    assert torch.equal(want, mm.int())
    assert torch.equal(d + s.table[M].int(), mg.int())
    if board in ((2, 2), (2, 3), (3, 2)):
        mini = solver_ref.MinimaxOutcome(*board)
        for (e, b2, t), o in zip(_host_state(eng, st), torch.sign(mg).cpu().numpy()):
            assert mini.outcome(e, b2, t) == o
    if board != (3, 4):
        eng.close()


SUPPORTED_TO_3X4 = [(1, k) for k in range(1, 11)] + [(k, 1) for k in range(2, 11)] + [(2, 2), (2, 3), (3, 2), (2, 4), (4, 2), (2, 5),
                                                                                       (5, 2), (3, 3), (3, 4), (4, 3)]


@pytest.mark.parametrize("board", SUPPORTED_TO_3X4)
def test_perfect_against_perfect(mods, board):
    """Random margin-optimal moves on both sides from the empty board: every position's outcome seen by player 0 and the
    final result equal the root outcome."""
    engine, solver, _ = mods
    if board in ((3, 4), (4, 3)):
        eng, s = _large(mods, board)
    else:
        eng, s = _solved(engine, solver, board)
    n = 64
    gen = torch.Generator(device=eng.device)
    gen.manual_seed(5)
    st = eng.new_states(n)
    root = int(s.outcome(st[:1])[0])
    for _ in range(s.E):
        res = eng.result(st)
        tp = st.view(torch.uint8).reshape(n, 32)[:, 20].long()
        o = s.outcome(st).long()
        assert bool((torch.where(tp == 0, o, -o) == root).all())
        opt = s.optimal_moves(st, "margin").double()
        live = res == 2
        mv = torch.multinomial(opt + (opt.sum(1, keepdim=True) == 0).double(), 1, generator=gen).reshape(-1)
        eng.play(st, torch.where(live, mv, torch.full_like(mv, -1)).int())
    res = eng.result(st).long()
    tp = st.view(torch.uint8).reshape(n, 32)[:, 20].long()
    assert bool((res != 2).all())
    assert bool((torch.where(tp == 0, res, -res) == root).all())
    if board not in ((3, 4), (4, 3)):
        eng.close()


def test_evaluator_rows(mods):
    engine, solver, _ = mods
    eng, s = _solved(engine, solver, (3, 3))
    st = _random_states(eng, 5000, seed=3)
    opt = s.optimal_moves(st, "outcome")
    k = opt.sum(1, keepdim=True).float()
    for mode, value in ((0, s.outcome(st).float()), (1, s.margin(st).float() / 9.0)):
        P = torch.full((5000, eng.A), 7.0, device=eng.device)
        V = torch.full((5000,), 7.0, device=eng.device)
        s.evaluate(eng, st, P, V, mode)
        assert torch.equal(P, torch.where(opt, 1.0 / k, torch.zeros_like(P)))
        assert torch.equal(V, value)
    with pytest.raises(ValueError):
        solver.SolverEvaluator(s, value="bogus")
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


@pytest.mark.parametrize("value", ["outcome", "margin"])
def test_evaluator_production_schedule_bit_exact(mods, value):
    """4096 trees of 3x3: eval cache + compact rows + adaptive ladder + device-driven loop == the plain wave loop."""
    engine, solver, _ = mods
    n, sims = 4096, 200
    plain = engine.Engine((3, 3), n_games=n, max_nodes=4 * sims + 64)
    s = solver.Solver(plain).solve()
    ev = solver.SolverEvaluator(s, value)
    roots = _random_states(plain, n, seed=7, max_depth=10)
    roots = torch.where((plain.result(roots) == 2).unsqueeze(1), roots, plain.new_states(n))
    ref = _search_moves(plain, ev, roots, sims, 2)
    info_plain = plain.status()
    eng = engine.Engine((3, 3), n_games=n, max_nodes=4 * sims + 64, eval_cache=16)
    eng.device_loop = True
    got = _search_moves(eng, ev, roots.clone(), sims, 2, graph_waves=4, adaptive=True)
    assert eng.device_loop
    info = eng.status()
    for m, (a, b) in enumerate(zip(ref, got)):
        for key in a:
            assert np.array_equal(a[key], b[key]), (value, m, key)
    assert info["sims"] == info_plain["sims"] and info["cache_hits"] > 0
    eng.close()
    plain.close()


def test_board_mismatch_and_unsolved(mods):
    engine, solver, _ = mods
    eng, s = _solved(engine, solver, (2, 2))
    other = engine.Engine((3, 3), n_games=4, max_nodes=64)
    with pytest.raises(ValueError):
        other.run_search(10, solver.SolverEvaluator(s))
    with pytest.raises(RuntimeError):
        solver.SolverEvaluator(solver.Solver(other))
    other.close()
    eng.close()


def _params(num_read=64, noise=(0.0, 0.0)):
    from dotsboxesaz_b200 import configuration
    p = copy.deepcopy(configuration.simple)
    p.self_play.mcts.mcts_num_read = num_read
    p.self_play.noise = noise
    return p


def test_play_games_async_and_grade_samples(mods):
    """Self-play with the solver as the net through play_games_async; grade_samples of the batch against NumPy."""
    engine, solver, solver_ref = mods
    from dotsboxesaz_b200 import samples, self_play
    n = 256
    eng = engine.Engine((3, 3), n_games=n, max_nodes=1024, eval_cache=14)
    s = solver.Solver(eng).solve()
    ev = solver.SolverEvaluator(s)
    bsp = self_play.BatchedSelfPlay(eng, ev, _params(64, (0.8, 0.25)), graph_waves=4, pending=1, adaptive=True)
    bsp.play_games_async(list(range(n)), seed=3)
    batch = samples.batch_from_selfplay(bsp, 0)
    assert len(batch) > n
    got = solver.grade_samples(s, batch)
    # NumPy: positions from the planes, margins from the host copy of the table
    g = solver_ref.Geometry(3, 3)
    T = s.table.cpu().numpy()
    x = batch.planes.cpu().numpy().astype(np.int64)
    pi = batch.pi.cpu().numpy().astype(np.float64)
    z = batch.z.cpu().numpy().astype(np.float64)
    P = g.plane
    rows = []
    for r in range(len(batch)):
        edges = sum(1 << a for a in range(2 * P) if x[r, a])
        k = int(np.int8(np.uint8(x[r, 2 * P])))
        other = 2 * g.LC - 2 * g.closed_boxes(edges) - k
        mm = solver_ref.move_margins(g, T, edges, (k, other), 0)
        fm = g.LC - k - g.closed_boxes(edges) + int(T[g.compact_mask(edges)])
        o = np.sign(fm)
        opt = np.zeros(eng.A, bool)
        for a, m in mm.items():
            opt[a] = np.sign(m) == o
        rows.append((opt[int(np.argmax(pi[r]))], float((pi[r] * opt).sum()), float(np.sign(z[r]) == o)))
    rows = np.array(rows, dtype=np.float64)
    assert got["n"] == len(batch)
    assert got["optimal_move_rate"] == pytest.approx(rows[:, 0].mean(), abs=1e-12)
    assert got["optimal_mass"] == pytest.approx(rows[:, 1].mean(), abs=1e-12)
    assert got["z_agreement"] == pytest.approx(rows[:, 2].mean(), abs=1e-12)
    # the rebuilt states carry the sample's key: the same rows as the recorded positions
    st = s.states_from_planes(batch.planes)
    assert torch.equal(eng.features(st, torch.int16).reshape(len(batch), -1).to(torch.uint8), batch.planes)
    eng.close()


def test_play_vs_solver(mods):
    engine, solver, solver_ref = mods
    n = 64
    eng = engine.Engine((3, 3), n_games=n, max_nodes=4096)
    s = solver.Solver(eng).solve()
    root = int(s.outcome(eng.new_states(1))[0])
    # the perfect model: no blunders, and the solver side never ends below its theoretical outcome.  Its moves are the
    # most visited ones (temperature 0.02 from the first move): the search gives every zero-prior move one exploratory
    # visit once the first visits of the optimal children have pushed their Q below 0 (a leaf's first backup adds
    # v + 1, mcts.py), so sampling in proportion to visits at temperature 1 can pick a losing move.
    params = _params()
    params.self_play.mcts.temperature = {0: 0.02}
    out = solver.play_vs_solver(eng, solver.SolverEvaluator(s), params, s, n, seed=1)
    assert out["blunders"] == 0 and out["model_moves"] > 0
    assert out["wins"] + out["draws"] + out["losses"] == n
    model_player = torch.arange(n, device=eng.device) % 2
    solver_theory = torch.where(model_player == 0, -root, root)
    assert bool((-out["result"].long() >= solver_theory).all())
    # a model that plays badly: the blunder count equals a host recount from the recorded moves
    out = solver.play_vs_solver(eng, engine.FakeNetEvaluator(0), _params(num_read=16), s, n - 3, seed=2)
    g = solver_ref.Geometry(3, 3)
    T = s.table.cpu().numpy()
    moves = out["moves"].cpu().numpy()
    model = out["model"].cpu().numpy()
    blunders = count = 0
    for p in range(moves.shape[0]):
        hs = _host_state(eng, out["states"][p].contiguous())
        for gi in np.flatnonzero(model[p]):
            edges, b2, tp = hs[gi]
            mm = solver_ref.move_margins(g, T, edges, b2, tp)
            o = np.sign(g.LC - b2[tp] - g.closed_boxes(edges) + int(T[g.compact_mask(edges)]))
            blunders += int(np.sign(mm[int(moves[p, gi])]) < o)
            count += 1
    assert count == out["model_moves"] and blunders == out["blunders"]
    assert out["blunders"] > 0
    eng.close()


@pytest.mark.parametrize("board", [(4, 4), (5, 5)])
def test_unsupported_boards_rejected(mods, board):
    engine, solver, _ = mods
    eng = engine.Engine(board, n_games=1, max_nodes=16)
    with pytest.raises(engine.EngineError, match="at most 32 edges"):
        solver.Solver(eng).solve()
    st = eng.new_states(1)
    buf = torch.zeros((1, eng.A), dtype=torch.int8, device=eng.device)
    assert eng.lib.dbaz_solver_moves(eng._h, None, engine._ptr(st), engine._ptr(buf), engine._ptr(buf), 1, eng._stream()) != 0
    assert b"at most 32 edges" in eng.lib.dbaz_last_error(eng._h)
    eng.close()


def test_wrong_table_size_rejected(mods):
    engine, solver, _ = mods
    eng = engine.Engine((3, 3), n_games=1, max_nodes=16)
    for n in (100, (1 << 24) - 1, 1 << 25):
        with pytest.raises(engine.EngineError, match="2\\^24"):
            solver.Solver(eng).solve(table=torch.empty((n,), dtype=torch.int8, device=eng.device))
    eng.close()
