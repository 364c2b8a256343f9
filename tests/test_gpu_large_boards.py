"""GPU: boards past 5x5 against the CPU oracle, bit for bit.  6x6 (A = 98), 6x7 (112), 7x7 (128), 4x7 (80) and the thin
1x31 / 31x1 (128) are the boards where the engine runs its widest instantiation (4 actions per lane, two 64-bit mask
words) and where actions 96..127 exist; 5x5 (3 actions per lane) and 1x1 are controls.  The oracle itself is pinned on
these boards by tests/test_oracle_large_boards.py.  Covered: the rule kernels (valid moves, play, result, features in
every dtype and layout, random rollouts), the batched search with 1..128 simulations in flight, the production
schedule (eval cache with split keys, compact rows, chains, overlap, adaptive ladder, device-driven loop) and device
self-play."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

BOARDS = [(6, 6), (7, 7), (6, 7), (4, 7), (1, 31), (31, 1), (5, 5), (1, 1)]


@pytest.fixture(scope="module")
def mods():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from dotsboxesaz_b200 import engine
    from oracle import oracle
    return engine, oracle


def _edges(eng, states_np):
    """packed states -> (bit a of the edge mask as uint8 [n, A], low word, high word)"""
    e = np.ascontiguousarray(states_np["edges"]).astype("<u8")
    bits = np.unpackbits(e.view(np.uint8).reshape(-1, 16), axis=1, bitorder="little")
    return bits[:, :eng.A], e[:, 0], e[:, 1]


def _padding(eng):
    a = np.arange(eng.A)
    plane = eng.rows * eng.cols
    p, rem = a // plane, a % plane
    l, c = rem // eng.cols, rem % eng.cols
    return np.where(p == 0, c == eng.C, l == eng.L)


def _cmp_states(eng, st, games, where):
    """Every field of the packed states against the oracle games: board bytes (the fixture record form), to_play,
    just_played, 2 * boxes_to_close and the 128-bit hash (hash_lo | hash_hi << 64 == the edge mask)."""
    h = eng.states_to_numpy(st)
    bits, lo, hi = _edges(eng, h)
    board = np.where(bits == 1, 255, np.where(_padding(eng), 1, 0)).astype(np.uint8)
    ref = np.stack([np.frombuffer(bytes(g.s.board)[:eng.A], np.uint8) for g in games])
    bad = np.flatnonzero((board != ref).any(1))
    assert bad.size == 0, (where, "board", int(bad[0]), np.flatnonzero(board[bad[0]] != ref[bad[0]]).tolist())
    assert np.array_equal(lo, np.array([g.s.hash_lo for g in games], np.uint64)), (where, "hash_lo")
    assert np.array_equal(hi, np.array([g.s.hash_hi for g in games], np.uint64)), (where, "hash_hi")
    assert np.array_equal(h["to_play"], [g.s.to_play for g in games]), (where, "to_play")
    assert np.array_equal(h["just_played"], [g.s.just_played for g in games]), (where, "just_played")
    assert np.array_equal(h["btc2"], [[g.s.btc2[0], g.s.btc2[1]] for g in games]), (where, "btc2")
    # the second hash word is boxes_to_close of the player to move, (0, 0) before the first move
    played = (lo | hi) != 0
    btc_tp = np.where(played, h["btc2"][np.arange(len(games)), h["to_play"]], 0)
    assert np.array_equal(btc_tp, [g.s.hash_btc2 for g in games]), (where, "hash[1]")
    return h


FEATURE_KINDS = [(dt, cl) for dt in ("int16", "float32", "bfloat16", "float16") for cl in (False, True)]


def _illegal(eng, og, g, ply, rng):
    """An illegal action of a kind that depends on (g, ply): -1, A, past A, a played edge, a padding cell, the last
    action (a padding cell on every board: 127 on 7x7)."""
    kind = (g + ply) % 6
    if kind == 0:
        return -1
    if kind == 1:
        return eng.A
    if kind == 2:
        return eng.A + 1 + int(rng.randint(0, 1 << 20))
    if kind == 3:
        played = np.flatnonzero(np.frombuffer(bytes(og.s.board)[:eng.A], np.uint8) == 255)
        if played.size:
            return int(played[rng.randint(played.size)])
        return -1
    if kind == 4:
        return int(rng.choice(np.flatnonzero(_padding(eng))))
    return eng.A - 1


@pytest.mark.parametrize("board", BOARDS)
def test_rules_vs_oracle(mods, board):
    """Several hundred random games to the end (host RNG), every ply: packed state and 128-bit hash, n_closed and the
    closed boxes, valid moves, result, features in all four dtypes and both layouts.  Illegal actions are thrown in
    along the way: they must give -1 and leave the state byte-equal."""
    engine, oracle = mods
    L, C = board
    n = 256
    eng = engine.Engine(board, n_games=1, max_nodes=4)
    try:
        assert eng.A == 2 * (L + 1) * (C + 1)
        rng = np.random.RandomState(L * 64 + C)
        games = [oracle.OracleGame(L, C) for _ in range(n)]
        st = eng.new_states(n)
        _cmp_states(eng, st, games, "init")
        n_edges = L * (C + 1) + C * (L + 1)
        illegal_seen = set()
        for ply in range(2 * n_edges + 4):  # a game that is handed an illegal action does not advance that ply
            mv = np.full(n, -1, np.int32)
            want_ncl = np.full(n, -1, np.int32)
            want_lc = np.full((n, 4), -1, np.int32)
            for g, og in enumerate(games):
                if og.result() is not None:
                    continue
                if (g + 3 * ply) % 11 == 0:
                    mv[g] = _illegal(eng, og, g, ply, rng)
                    illegal_seen.add((g + ply) % 6)
                    continue
                mv[g] = int(rng.choice(np.flatnonzero(og.valid_moves())))
                closed = og.play_(int(mv[g]))
                want_ncl[g] = len(closed)
                for j, (l, c) in enumerate(closed):
                    want_lc[g, 2 * j:2 * j + 2] = (l, c)
            before = eng.states_to_numpy(st)
            ncl, lc = eng.play(st, mv)
            where = (board, ply)
            ncl, lc = ncl.cpu().numpy(), lc.cpu().numpy()
            bad = np.flatnonzero(ncl != want_ncl)
            assert bad.size == 0, (where, "n_closed", int(bad[0]), int(mv[bad[0]]), int(ncl[bad[0]]), int(want_ncl[bad[0]]))
            bad = np.flatnonzero((lc != want_lc).any(1))
            assert bad.size == 0, (where, "closed_lc", int(bad[0]), int(mv[bad[0]]), lc[bad[0]].tolist(), want_lc[bad[0]].tolist())
            h = _cmp_states(eng, st, games, where)
            # a rejected action leaves all 32 bytes of the state as they were
            rej = want_ncl < 0
            assert np.array_equal(h[rej].view(np.uint8), before[rej].view(np.uint8)), (where, "rejected move changed the state")
            valid = eng.valid_moves(st).cpu().numpy()
            ref_valid = np.stack([og.valid_moves() for og in games])
            bad = np.flatnonzero((valid != ref_valid).any(1))
            assert bad.size == 0, (where, "valid", int(bad[0]), np.flatnonzero(valid[bad[0]] != ref_valid[bad[0]]).tolist())
            res = eng.result(st).cpu().numpy()
            assert np.array_equal(res, [2 if og.result() is None else og.result() for og in games]), (where, "result")
            ref_f = np.stack([og.features() for og in games]).astype(np.float32)
            for dt, cl in FEATURE_KINDS:
                f = eng.features(st, getattr(torch, dt), cl)
                assert f.shape == (n, 3, L + 1, C + 1)
                f = f.float().cpu().numpy()
                bad = np.flatnonzero((f != ref_f).reshape(n, -1).any(1))
                assert bad.size == 0, (where, "features", dt, "NHWC" if cl else "NCHW", int(bad[0]))
            if all(og.result() is not None for og in games):
                break
        assert all(og.result() is not None for og in games)
        assert illegal_seen == set(range(6)) or n_edges < 6
    finally:
        eng.close()


@pytest.mark.parametrize("board", BOARDS)
def test_random_rollouts_vs_oracle(mods, board):
    """Random playouts with the game counter across and above 2^32 (both words of the 64-bit counter feed the RNG):
    number of plies, move list, final state and result of every third game."""
    engine, oracle = mods
    L, C = board
    eng = engine.Engine(board, n_games=1, max_nodes=4)
    try:
        for game0 in ((1 << 32) - 300, (7 << 32) + 12345):
            n = 600
            st = eng.new_states(n)
            plies, moves = eng.random_rollout(st, seed=0x5EED0000BEEF, game0=game0, record_moves=True)
            plies, moves = plies.cpu().numpy(), moves.cpu().numpy()
            res = eng.result(st).cpu().numpy()
            idx = list(range(0, n, 3))
            games = []
            for g in idx:
                og = oracle.OracleGame(L, C)
                mv = og.random_rollout(0x5EED0000BEEF, game0 + g)
                assert plies[g] == len(mv) and moves[g][:len(mv)].tolist() == mv, (board, game0, g)
                assert int(res[g]) == og.record()["result"] != 2, (board, game0, g)
                games.append(og)
            _cmp_states(eng, st[idx], games, (board, game0))
    finally:
        eng.close()


def _roots(eng, oracle, n, rng, max_frac=0.8):
    """n seeded start positions 0 .. max_frac * n_edges plies deep, played on the engine and on oracle games."""
    L, C = eng.L, eng.C
    n_edges = L * (C + 1) + C * (L + 1)
    depth = rng.randint(0, max(1, int(max_frac * n_edges)) + 1, n)
    depth[:2] = 0  # an empty board among them
    og = [oracle.OracleGame(L, C) for _ in range(n)]
    st = eng.new_states(n)
    for ply in range(int(depth.max())):
        mv = np.full(n, -1, np.int32)
        for g in range(n):
            if ply < depth[g] and og[g].result() is None:
                mv[g] = rng.choice(np.flatnonzero(og[g].valid_moves()))
                og[g].play_(int(mv[g]))
        eng.play(st, mv)
    return st, og


def _snapshot(eng):
    vis = eng.root_visits().cpu().numpy()
    W, P, S, U = (x.cpu().numpy() for x in eng.root_children())
    st, rW, q = (x.cpu().numpy() for x in eng.tree_stats())
    return {"visits": vis, "W": W, "priors": P, "sign": S, "ucb": U, "stats": st, "root_W": rW, "q": q}


def _check_tree(eng, snap, g, tree, where):
    """Root of tree g of the engine against the oracle tree, bit for bit."""
    r = tree.root()
    assert np.array_equal(snap["visits"][g], r["visits"]), (where, "visits", g, np.flatnonzero(snap["visits"][g] != r["visits"]).tolist())
    assert np.array_equal(snap["W"][g].view(np.uint32), r["W"].view(np.uint32)), (where, "W", g)
    assert np.array_equal(snap["priors"][g].view(np.uint64), r["priors"].view(np.uint64)), (where, "priors", g)
    assert np.array_equal(snap["ucb"][g].view(np.uint64), r["ucb"].view(np.uint64)), (where, "ucb", g)
    v = r["visits"] > 0
    assert np.array_equal(snap["sign"][g][v], r["sign"][v]), (where, "sign", g)
    st = snap["stats"][g]
    assert [int(x) for x in st[:4]] == [r["root_N"]] + r["stats"][:3], (where, "stats", g, st[:4].tolist(), r["root_N"], r["stats"])
    assert (bool(st[4]), bool(st[5])) == (r["is_expanded"], r["is_terminal"]), (where, "flags", g)
    assert np.float32(snap["root_W"][g]).view(np.uint32) == np.float32(r["root_W"]).view(np.uint32), (where, "root_W", g)
    assert np.float32(snap["q"][g]).view(np.uint32) == np.float32(r["stats"][3]).view(np.uint32), (where, "q", g)
    return r


def _check_root_states(eng, trees, where):
    _cmp_states(eng, eng.root_states(), [t.root()["state"] for t in trees], where)


def _pick_moves(trees, move_i):
    """The next move of every tree: the most visited child, a legal child chosen by position (often unvisited), or one
    of the highest legal actions (>= 96 where the board has them).  -1 for terminal roots."""
    moves = np.full(len(trees), -1, np.int32)
    for g, t in enumerate(trees):
        r = t.root()
        if r["is_terminal"]:
            continue
        legal = np.flatnonzero(r["state"].valid_moves())
        if g % 3 == 1:
            moves[g] = int(np.argmax(r["visits"]))
        elif g % 3 == 2:
            moves[g] = int(legal[-1 - (move_i % len(legal))])
        else:
            moves[g] = int(legal[(g + move_i) % len(legal)])
    return moves


@pytest.mark.parametrize("kind", [0, 1])
@pytest.mark.parametrize("pending", [1, 8, 128])
@pytest.mark.parametrize("board", [(6, 6), (7, 7), (6, 7), (1, 31), (5, 5)])
def test_batched_search_vs_oracle(mods, board, pending, kind):
    """Many trees in lock-step from seeded positions, Dirichlet noise, four moves with tree reuse (onto the most visited
    child, onto unvisited children, onto the highest actions), plain and graph-captured wave loops, 1, 8 and 128
    simulations in flight (128 = A on 7x7: the first wave is min(K, A) wide).  Visits, W, priors, UCB bits, the sign of
    visited children, the tree statistics, root W and q and the root state equal the oracle's."""
    engine, oracle = mods
    n, sims = 40, 200
    eng = engine.Engine(board, n_games=n, max_nodes=4096, max_pending=pending)
    try:
        rng = np.random.RandomState(board[0] * 1000 + board[1] * 10 + pending + kind)
        st, og = _roots(eng, oracle, n, rng)
        trees = [oracle.OracleTree(*board, og[g].s, kind=kind) for g in range(n)]
        eng.reset_roots(st)
        ev = engine.FakeNetEvaluator(kind)
        checked = 0
        for move_i in range(4):
            reads = np.array([sims if g % 5 else sims // 2 + 7 for g in range(n)], np.int32)
            term = np.array([t.root()["is_terminal"] for t in trees])
            reads[term] = -1
            valid = np.stack([t.root()["state"].valid_moves() for t in trees])
            noise = rng.dirichlet(np.ones(eng.A) * 0.8, size=n) * valid
            eng.run_search(torch.from_numpy(reads), ev, noise=torch.from_numpy(noise), coeff=0.25, max_reads=sims,
                           pending=pending, graph_waves=8 if move_i % 2 else 0)
            snap = _snapshot(eng)
            for g in range(n):
                if term[g]:
                    continue
                trees[g].search(int(reads[g]), noise=noise[g], coeff=0.25, max_pending=pending)
                _check_tree(eng, snap, g, trees[g], (board, pending, kind, move_i))
                checked += 1
            _check_root_states(eng, trees, (board, pending, kind, move_i, "root"))
            moves = _pick_moves(trees, move_i)
            for g in range(n):
                if moves[g] >= 0:
                    trees[g].reroot(int(moves[g]), True)
            eng.advance_roots(moves, reuse=True)
            assert eng.status()["errors"] == 0
        _check_root_states(eng, trees, (board, pending, kind, "after the last re-root"))
        assert checked > 3 * n
    finally:
        eng.close()


@pytest.mark.parametrize("board,device_loop", [((6, 6), True), ((7, 7), True), ((7, 7), False), ((6, 6), False)])
def test_production_schedule_vs_oracle(mods, board, device_loop):
    """The schedule self-play runs with -- eval cache (keys split across cells past 88 actions), compact rows, in-kernel
    chains bounded by count and time, the adaptive batch ladder, driven by the device's WHILE/SWITCH loop or by the
    host -- checked tree by tree against the oracle itself."""
    engine, oracle = mods
    n, sims = 128, 150
    eng = engine.Engine(board, n_games=n, max_nodes=4 * sims + 64, eval_cache=12)
    try:
        eng.set_mode(False, 2)
        eng.device_loop = device_loop
        rng = np.random.RandomState(17 + board[0])
        st, og = _roots(eng, oracle, n, rng, max_frac=0.6)
        trees = [oracle.OracleTree(*board, og[g].s) for g in range(n)]
        eng.reset_roots(st)
        ev = engine.FakeNetEvaluator(0)
        for move_i in range(3):
            reads = np.array([sims if g % 7 else sims // 3 for g in range(n)], np.int32)
            term = np.array([t.root()["is_terminal"] for t in trees])
            reads[term] = -1
            valid = np.stack([t.root()["state"].valid_moves() for t in trees])
            noise = rng.dirichlet(np.ones(eng.A) * 0.8, size=n) * valid
            eng.run_search(torch.from_numpy(reads), ev, noise=torch.from_numpy(noise), coeff=0.25, graph_waves=4, adaptive=True)
            snap = _snapshot(eng)
            for g in range(n):
                if term[g]:
                    continue
                trees[g].search(int(reads[g]), noise=noise[g], coeff=0.25)
                _check_tree(eng, snap, g, trees[g], (board, device_loop, move_i))
            moves = _pick_moves(trees, move_i)
            for g in range(n):
                if moves[g] >= 0:
                    trees[g].reroot(int(moves[g]), True)
            eng.advance_roots(moves, reuse=True)
        _check_root_states(eng, trees, (board, device_loop, "root"))
        info = eng.status()
        assert info["errors"] == 0 and info["cache_hits"] > 0
        assert eng.device_loop == device_loop       # the conditional graph was built, not replaced by the host loop
        assert eng.wave_counts() == (0, 0)
    finally:
        eng.close()


@pytest.mark.parametrize("mode", ["device", "async"])
@pytest.mark.parametrize("board,num_read", [((6, 6), 96), ((7, 7), 64)])
def test_device_selfplay_vs_oracle(mods, board, num_read, mode):
    """play_games_device / play_games_async on the large boards (k_selfplay_pick and k_selfplay_restart at 4 actions per
    lane, the pre-drawn noise rows, the draw of the move): 64 games, 20 of them replayed on the oracle."""
    from test_gpu_selfplay_parity import _params, _replay_device_history
    from dotsboxesaz_b200 import self_play
    engine, _ = mods
    n = 64
    eng = engine.Engine(board, n_games=n, max_nodes=4096, eval_cache=14)
    try:
        bsp = self_play.BatchedSelfPlay(eng, engine.FakeNetEvaluator(0), _params(num_read), graph_waves=8 if mode == "device" else 4)
        assert bsp.adaptive and bsp.pending == 1
        info = (bsp.play_games_device if mode == "device" else bsp.play_games_async)(range(n), seed=23)
        assert info["errors"] == 0
        games = list(range(0, n, 3))[:20]
        searches, sims = _replay_device_history(bsp, board, num_read, games)
        n_edges = board[0] * (board[1] + 1) + board[1] * (board[0] + 1)
        assert searches >= len(games) * n_edges // 2
        # the moves cover the second mask word, and on 7x7 the actions past 95 (on 6x6 these are padding cells)
        moves = torch.stack(bsp._device_hist["moves"]).cpu().numpy()
        assert (moves >= 64).any() and ((moves >= 96).any() or board == (6, 6))
    finally:
        eng.close()
