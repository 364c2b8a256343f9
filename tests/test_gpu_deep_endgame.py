"""GPU: the deep tier of the exact endgame solver (positions with 17 <= f <= 32 free edges, DeepEndgameSolver and
dbaz_endgame_deep_moves).  Byte for byte against the 32-edge table on 3x4, 4x3 and 2x6 for every f from 17 to E, with one
position per pass and with large passes; against endgame_numpy on the large boards; by the one-step recurrence across
tiers up to f = 32; mixed batches; grading and the perfect opponent against the full-table Solver; the error paths."""
import copy

import numpy as np
import pytest

import endgame_ref
from test_gpu_endgame import _mask_states, _real_actions, _rollout_states

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

GEOM = 512  # workspace bytes of one position's geometry, beside its 2^f table


@pytest.fixture(scope="module")
def mods():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from dotsboxesaz_b200 import endgame, engine, solver
    from oracle import solver_ref
    return engine, solver, endgame, solver_ref


def _states_at(eng, f, n, gen):
    """n states with exactly f free edges: half random masks, half rollouts of E - f plies"""
    E = len(_real_actions(eng.L, eng.C))
    k = n // 2
    parts = [_mask_states(eng, f, n - k, gen)]
    if k:
        parts.append(_rollout_states(eng, torch.full((k,), E - f, dtype=torch.int64, device=eng.device), gen))
    return torch.cat(parts).contiguous()


def _per_f(f):
    return 256 if f <= 24 else 16 if f <= 28 else 2


@pytest.mark.parametrize("board", [(3, 4), (4, 3), (2, 6)])
def test_deep_equals_32_edge_table(mods, board):
    """Every f in 17 .. E (the empty board included): DeepEndgameSolver(eng, 32).moves == Solver.moves byte for byte, with
    an 8 GiB workspace and with a workspace of exactly one position."""
    engine, solver, endgame, _ = mods
    eng = engine.Engine(board, n_games=1, max_nodes=16)
    s = solver.Solver(eng).solve()
    E = s.E
    gen = torch.Generator(device=eng.device)
    gen.manual_seed(board[0] * 13 + board[1])
    st = torch.cat([_states_at(eng, f, _per_f(f), gen) for f in range(17, E + 1)] + [eng.new_states(1)]).contiguous()
    mm, mg = s.moves(st)
    big = endgame.DeepEndgameSolver(eng, 32, workspace_bytes=8 << 30)
    f = big.free_edges(st)
    assert int(f.min()) == 17 and int(f.max()) == E
    emm, emg = big.moves(st)
    assert torch.equal(emm, mm) and torch.equal(emg, mg)
    assert bool(big.solvable(st).all())
    del big
    for fv in range(17, E + 1):
        rows = (f == fv).nonzero().reshape(-1)
        one = endgame.DeepEndgameSolver(eng, fv, workspace_bytes=(1 << fv) + GEOM)
        omm, omg = one.moves(st[rows].contiguous())
        assert torch.equal(omm, mm[rows]) and torch.equal(omg, mg[rows]), (board, fv)
        del one
    del s
    eng.close()
    torch.cuda.empty_cache()


def _host_rows(eng, st):
    rec = eng.states_to_numpy(st)
    return [(int(r["edges"][0]) | (int(r["edges"][1]) << 64), (int(r["btc2"][0]), int(r["btc2"][1])), int(r["to_play"])) for r in rec]


@pytest.mark.parametrize("board", [(4, 4), (5, 5), (7, 7), (1, 31), (31, 1)])
def test_large_boards_equal_numpy(mods, board):
    """Move margins and final margins against endgame_numpy, f = 17 .. 20, a mask and a rollout state each."""
    engine, _, endgame, solver_ref = mods
    eng = engine.Engine(board, n_games=1, max_nodes=16)
    gen = torch.Generator(device=eng.device)
    gen.manual_seed(board[0] * 41 + board[1])
    st = torch.cat([_states_at(eng, f, 2, gen) for f in range(17, 21)]).contiguous()
    deep = endgame.DeepEndgameSolver(eng, 20)
    mm, mg = (x.cpu().numpy() for x in deep.moves(st))
    g = solver_ref.Geometry(*board)
    high = 0
    for r, (edges, btc2, tp) in enumerate(_host_rows(eng, st)):
        want_mm, want_final = endgame_ref.endgame_moves(g, edges, btc2, tp)
        assert np.array_equal(mm[r].astype(np.int64), want_mm), (board, r)
        assert int(mg[r]) == want_final, (board, r)
        high += int((want_mm[64:] != -128).any())
    assert high > 0 or g.A <= 64
    eng.close()


def _check_recurrence(eng, deep, st):
    """mm[s][a] == (a closes a box ? mg[s a] : -mg[s a]) for every free action a, with the successor from Engine.play and
    its margin from the same solver; mg[s] == max_a mm[s][a].  The recurrence holds for states whose scores add up as in
    a played game (btc2[0] + btc2[1] = 2 LC - 2 closed), so the states are first rebuilt from their feature planes, which
    keep the edges and btc2[to_play] and derive the other score from that sum."""
    n = st.shape[0]
    st = deep.states_from_planes(eng.features(st, torch.int16).reshape(n, -1)).contiguous()
    mm, mg = deep.moves(st)
    valid = mm != -128
    assert torch.equal(valid.sum(1), deep.free_edges(st))
    rows, acts = valid.nonzero(as_tuple=True)
    succ = st[rows].clone()
    n_closed, _ = eng.play(succ, acts.int())
    smg = deep.margin(succ).long()
    assert bool((smg != -128).all())
    want = torch.where(n_closed > 0, smg, -smg)
    assert torch.equal(mm[rows, acts].long(), want)
    best = torch.where(valid, mm.long(), torch.full_like(mm, -128).long()).max(1).values
    assert torch.equal(best, mg.long())


@pytest.mark.parametrize("board", [(5, 5), (7, 7)])
def test_recurrence_across_tiers(mods, board):
    """f = 17 .. 28: each f checked against the solver's own f - 1 (at f = 17 the shared-memory tier)."""
    engine, _, endgame, _ = mods
    eng = engine.Engine(board, n_games=1, max_nodes=16)
    gen = torch.Generator(device=eng.device)
    gen.manual_seed(board[0] * 7 + 1)
    deep = endgame.DeepEndgameSolver(eng, 28)
    for f in range(17, 29):
        _check_recurrence(eng, deep, _states_at(eng, f, 4 if f <= 24 else 2, gen))
    eng.close()
    torch.cuda.empty_cache()


def test_recurrence_at_32_free_edges(mods):
    """4x4 after 8 plies (f = 32) against its successors at f = 31."""
    engine, _, endgame, _ = mods
    eng = engine.Engine((4, 4), n_games=1, max_nodes=16)
    gen = torch.Generator(device=eng.device)
    gen.manual_seed(32)
    deep = endgame.DeepEndgameSolver(eng, 32)
    st = _states_at(eng, 32, 2, gen)
    assert bool((deep.free_edges(st) == 32).all())
    _check_recurrence(eng, deep, st)
    eng.close()
    torch.cuda.empty_cache()


def test_mixed_batch(mods):
    """5x5, rows with f <= 16, 17 .. 20 and > 20 shuffled: the first equal EndgameSolver(eng, 16), the deep rows equal
    per-f calls, the rest are all ILLEGAL; the inherited queries follow."""
    engine, _, endgame, _ = mods
    eng = engine.Engine((5, 5), n_games=1, max_nodes=16)
    gen = torch.Generator(device=eng.device)
    gen.manual_seed(5)
    st = torch.cat([_states_at(eng, f, 6, gen) for f in (0, 5, 10, 12, 16, 17, 18, 19, 20, 21, 24, 40, 60)])
    st = st[torch.randperm(st.shape[0], generator=gen, device=eng.device)].contiguous()
    deep = endgame.DeepEndgameSolver(eng, 20)
    mm, mg = deep.moves(st)
    f = deep.free_edges(st)
    low, mid, high = f <= 16, (f >= 17) & (f <= 20), f > 20
    smm, smg = endgame.EndgameSolver(eng, 16).moves(st)
    assert torch.equal(mm[low], smm[low]) and torch.equal(mg[low], smg[low])
    for fv in range(17, 21):
        rows = (f == fv).nonzero().reshape(-1)
        omm, omg = deep.moves(st[rows].contiguous())
        assert torch.equal(mm[rows], omm) and torch.equal(mg[rows], omg)
        assert bool((omg != -128).all())
    assert bool((mm[high] == -128).all()) and bool((mg[high] == -128).all())
    assert torch.equal(deep.solvable(st), low | mid)
    assert torch.equal(deep.margin(st), mg)
    assert torch.equal(deep.outcome(st), torch.where(mg == -128, mg, torch.sign(mg)))
    assert torch.equal(deep.optimal_moves(st, "margin"), (mm != -128) & (mm == mg.unsqueeze(1)))
    eng.close()


def _params(num_read=64, noise=(0.0, 0.0)):
    from dotsboxesaz_b200 import configuration
    p = copy.deepcopy(configuration.simple)
    p.self_play.mcts.mcts_num_read = num_read
    p.self_play.noise = noise
    return p


def test_grade_samples_3x4(mods):
    """A 3x4 self-play batch graded with DeepEndgameSolver(eng, 32) gives the full-table Solver's figures exactly."""
    engine, solver, endgame, _ = mods
    from dotsboxesaz_b200 import samples, self_play
    n = 32
    eng = engine.Engine((3, 4), n_games=n, max_nodes=1024, eval_cache=14)
    bsp = self_play.BatchedSelfPlay(eng, engine.FakeNetEvaluator(0), _params(32, (0.8, 0.25)), graph_waves=4, pending=1, adaptive=True)
    bsp.play_games_async(list(range(n)), seed=11)
    batch = samples.batch_from_selfplay(bsp, 0)
    got = solver.grade_samples(endgame.DeepEndgameSolver(eng, 32), batch)
    s = solver.Solver(eng).solve()
    want = solver.grade_samples(s, batch)
    assert got.pop("n_solved") == got["n"] == len(batch)
    assert got == want
    del s
    eng.close()
    torch.cuda.empty_cache()


def _start(eng, depth, n, gen):
    """n games still going on after `depth` random plies"""
    st = _rollout_states(eng, torch.full((4 * n,), depth, dtype=torch.int64, device=eng.device), gen)
    st = st[eng.result(st) == 2][:n].contiguous()
    assert st.shape[0] == n
    return st


def test_play_vs_solver_from_mid_game_3x4(mods):
    """From mid-game start states the deep tier is the same perfect opponent as the full table: identical outputs."""
    engine, solver, endgame, _ = mods
    n = 16
    eng = engine.Engine((3, 4), n_games=n, max_nodes=4096)
    gen = torch.Generator(device=eng.device)
    gen.manual_seed(12)
    start = torch.cat([_start(eng, 10, n // 2, gen), _start(eng, 14, n // 2, gen)])
    s = solver.Solver(eng).solve()
    outs = [solver.play_vs_solver(eng, engine.FakeNetEvaluator(0), _params(16), sv, n, seed=4, start_states=start)
            for sv in (s, endgame.DeepEndgameSolver(eng, 32))]
    a, b = outs
    assert a["model_moves"] > 0
    for key in a:
        if isinstance(a[key], torch.Tensor):
            assert torch.equal(a[key], b[key]), key
        else:
            assert a[key] == b[key], key
    assert torch.equal(a["states"][0][:, :2], start[:, :2])
    del s
    eng.close()
    torch.cuda.empty_cache()


def test_play_vs_solver_4x4(mods):
    """4x4 from positions with f <= 22: the model never ends above the start position's outcome from its side."""
    engine, solver, endgame, _ = mods
    n = 32
    eng = engine.Engine((4, 4), n_games=n, max_nodes=4096)
    gen = torch.Generator(device=eng.device)
    gen.manual_seed(44)
    start = torch.cat([_start(eng, 18, n // 2, gen), _start(eng, 22, n // 2, gen)])
    deep = endgame.DeepEndgameSolver(eng, 22)
    assert bool(deep.solvable(start).all())
    o = deep.outcome(start).long()
    to_play = start.view(torch.uint8).reshape(n, 32)[:, 20].long()
    model_player = torch.arange(n, device=eng.device) % 2
    bound = torch.where(to_play == model_player, o, -o)
    out = solver.play_vs_solver(eng, engine.FakeNetEvaluator(0), _params(16), deep, n, seed=5, start_states=start)
    assert out["model_moves"] > 0 and out["wins"] + out["draws"] + out["losses"] == n
    assert bool((out["result"].long() <= bound).all())
    eng.close()


def test_error_paths(mods):
    engine, solver, endgame, _ = mods
    eng = engine.Engine((5, 5), n_games=2, max_nodes=16)
    gen = torch.Generator(device=eng.device)
    gen.manual_seed(2)
    for mf in (16, 33):
        with pytest.raises(ValueError, match="max_free must be in"):
            endgame.DeepEndgameSolver(eng, mf)
    with pytest.raises(ValueError, match="workspace bytes"):
        endgame.DeepEndgameSolver(eng, 20, workspace_bytes=1 << 20)
    deep = endgame.DeepEndgameSolver(eng, 20)
    st = eng.new_states(1)
    P = torch.zeros((1, eng.A), device=eng.device)
    V = torch.zeros((1,), device=eng.device)
    with pytest.raises(ValueError):
        deep.evaluate(eng, st, P, V)
    with pytest.raises(ValueError):
        deep.adjudicate(None, None)
    with pytest.raises(ValueError):
        endgame.EndgameEvaluator(engine.FakeNetEvaluator(0), deep)
    with pytest.raises(ValueError, match="max_free"):
        solver.play_vs_solver(eng, engine.FakeNetEvaluator(0), _params(16), deep, 2, start_states=eng.new_states(2))

    # the C ABI
    good = _states_at(eng, 17, 3, gen)
    ws = torch.empty(((1 << 17) + GEOM,), dtype=torch.int8, device=eng.device)
    mm = torch.empty((3, eng.A), dtype=torch.int8, device=eng.device)
    mg = torch.empty((3,), dtype=torch.int8, device=eng.device)
    p = engine._ptr

    def call(states=good, n=3, f=17, workspace=ws, nbytes=ws.numel(), move_margin=mm, margin=mg):
        return eng.lib.dbaz_endgame_deep_moves(eng._h, p(states), n, f, p(workspace), nbytes, p(move_margin), p(margin), eng._stream())

    def valid_call_works():
        assert call() == 0
        want_mm, want_mg = endgame.DeepEndgameSolver(eng, 17).moves(good)
        assert torch.equal(mm, want_mm) and torch.equal(mg, want_mg)

    mixed = torch.cat([good[:1], _states_at(eng, 18, 2, gen)]).contiguous()
    rejections = [
        (dict(f=16), "dbaz_endgame_deep_moves: f must be in [17, 32], got 16"),
        (dict(f=33), "dbaz_endgame_deep_moves: f must be in [17, 32], got 33"),
        (dict(nbytes=(1 << 17) + GEOM - 1),
         "dbaz_endgame_deep_moves: one position with f = 17 needs 2^17 + 512 = 131584 workspace bytes, got 131583"),
        (dict(states=None), "dbaz_endgame_deep_moves: null buffer"),
        (dict(workspace=None), "dbaz_endgame_deep_moves: null buffer"),
        (dict(move_margin=None), "dbaz_endgame_deep_moves: null buffer"),
        (dict(margin=None), "dbaz_endgame_deep_moves: null buffer"),
        (dict(n=-1), "dbaz_endgame_deep_moves: n must be >= 0, got -1"),
        (dict(states=mixed), "dbaz_endgame_deep_moves: 2 of 3 states do not have f = 17 free edges"),
    ]
    for kw, msg in rejections:
        assert call(**kw) != 0, msg
        assert eng.lib.dbaz_last_error(eng._h).decode() == msg
        valid_call_works()
    assert call(n=0) == 0
    with pytest.raises(engine.EngineError, match="do not have f = 17"):
        eng._ck(call(states=mixed))
    eng.close()
