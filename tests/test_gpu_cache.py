"""GPU: the eval cache (utils/proxies.py:23-26,35-43), compact leaf rows and the adaptive wave loop change the
schedule of a lock-step search, never its result.  Every test runs the same searches twice -- plain (row == tree,
fixed wave count, no cache) and with the feature under test -- through the C ABI and compares visit counts, W,
priors, UCB and tree statistics bit for bit; one of the runs is also checked against the CPU oracle."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def mods():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from dotsboxesaz_b200 import engine
    from oracle import oracle
    return engine, oracle


def _roots(eng, n, max_plies, seed):
    """n random legal positions 0..max_plies plies deep (host RNG, engine rules)."""
    rng = np.random.RandomState(seed)
    st = eng.new_states(n)
    depth = rng.randint(0, max_plies + 1, n)
    played = [[] for _ in range(n)]
    for ply in range(max_plies):
        valid = eng.valid_moves(st).cpu().numpy()
        mv = np.full(n, -1, np.int32)
        for g in range(n):
            if depth[g] > ply and valid[g].any():
                mv[g] = rng.choice(np.flatnonzero(valid[g]))
                played[g].append(int(mv[g]))
        eng.play(st, mv)
    return st, played


def _snapshot(eng):
    vis = eng.root_visits().cpu().numpy()
    W, P, S, U = (x.cpu().numpy() for x in eng.root_children())
    st, rW, q = (x.cpu().numpy() for x in eng.tree_stats())
    return {"visits": vis, "W": W, "priors": P, "ucb": U, "stats": st[:, :7], "root_W": rW, "q": q}


def _same(a, b, where):
    for k in a:
        assert np.array_equal(a[k].view(np.uint8) if a[k].dtype.kind == "f" else a[k],
                              b[k].view(np.uint8) if b[k].dtype.kind == "f" else b[k]), (where, k)


def _play(eng, ev, roots, sims, moves, noise_seed, **kw):
    """`moves` searches with re-roots onto the most visited child; returns the per-move snapshots."""
    rng = np.random.RandomState(noise_seed)
    eng.reset_roots(roots)
    out = []
    for m in range(moves):
        valid = eng.valid_moves(eng.root_states()).cpu().numpy()
        noise = rng.dirichlet(np.ones(eng.A) * 0.8, size=eng.n_games) * valid
        eng.run_search(sims, ev, noise=torch.from_numpy(noise), coeff=0.25, **kw)
        snap = _snapshot(eng)
        out.append(snap)
        mv = np.where(snap["visits"].sum(1) > 0, snap["visits"].argmax(1), -1).astype(np.int32)
        eng.advance_roots(mv, reuse=True)
    return out


@pytest.mark.parametrize("device_loop", [True, False], ids=["device_loop", "host_loop"])
@pytest.mark.parametrize("board,n,sims,log2,max_inline,margin", [((3, 3), 192, 300, 14, 0, 1.125), ((3, 3), 192, 300, 5, 2, 1.125),
                                                                 ((5, 5), 96, 200, 12, 0, 1.125), ((2, 3), 64, 150, 10, 3, 1.125),
                                                                 ((3, 3), 512, 300, 14, 4, 0.4), ((5, 5), 256, 200, 12, 2, 0.25)])
def test_cache_compact_adaptive_bit_exact(mods, board, n, sims, log2, max_inline, margin, device_loop):
    """margin < 1 sizes the evaluator's batch BELOW what the waves ask for, so leaves overflow the batch all the time and
    their selections are dropped and repeated (dbaz_search_set_batch_rows).  device_loop: the adaptive loop as one
    conditional graph per search, or driven by the host (the fallback where a driver cannot build that graph)."""
    engine, oracle = mods
    ev = engine.FakeNetEvaluator(0)
    plain = engine.Engine(board, n_games=n, max_nodes=4 * sims + 64)
    roots, played = _roots(plain, n, 10, seed=7)
    ref = _play(plain, ev, roots, sims, 4, noise_seed=3)
    info_plain = plain.status()
    plain.close()

    eng = engine.Engine(board, n_games=n, max_nodes=4 * sims + 64, eval_cache=log2)
    eng.set_mode(False, max_inline)
    eng.ROW_MARGIN = margin
    eng.device_loop = device_loop
    got = _play(eng, ev, roots.clone(), sims, 4, noise_seed=3, graph_waves=4, adaptive=True)
    assert eng.device_loop == device_loop  # the conditional graph was built, not replaced by the host loop
    info = eng.status()
    for m, (a, b) in enumerate(zip(ref, got)):
        _same(a, b, (board, "move", m))
    assert info["sims"] == info_plain["sims"] and info["path_nodes"] == info_plain["path_nodes"]
    assert info["cache_hits"] > 0
    assert info_plain["cache_hits"] == 0
    assert eng.wave_counts() == (0, 0)
    # fewer waves than simulations: hits and terminal leaves finished inside the step kernel
    if margin >= 1:
        assert eng.n_waves < 4 * (sims + 2) + 4 * 16
    else:
        assert eng.n_waves > 4 * (sims + 2)  # leaves did overflow the undersized batches and were repeated

    # the cached engine without the adaptive loop (row == tree, fixed wave count) gives the same result again
    eng.clear_eval_cache()
    got2 = _play(eng, ev, roots.clone(), sims, 2, noise_seed=3, graph_waves=0)
    for m, (a, b) in enumerate(zip(ref[:2], got2)):
        _same(a, b, (board, "fixed loop, move", m))
    eng.close()

    # one tree of the run against the CPU oracle
    L, C = board
    g = 5
    game = oracle.OracleGame(L, C)
    for mv in played[g]:
        game.play_(mv)
    tree = oracle.OracleTree(L, C, game.s)
    rng = np.random.RandomState(3)
    for m in range(2):
        if game.result() is not None:
            break
        # the engine drew the noise of all games of a move at once: reproduce the stream, keep row g
        noise = rng.dirichlet(np.ones(tree.A) * 0.8, size=n)[g] * game.valid_moves()
        vis = tree.search(sims, noise=noise, coeff=0.25)
        assert np.array_equal(vis, got[m]["visits"][g]), ("oracle", m)
        mv = int(np.argmax(vis))
        tree.reroot(mv, True)
        game.play_(mv)


def test_cache_persists_across_searches_and_clear(mods):
    """Second identical search from the same roots is served from the table; after clear it is not."""
    engine, _ = mods
    n, sims = 128, 200
    eng = engine.Engine((3, 3), n_games=n, max_nodes=sims + 16, eval_cache=20)  # 40 slots per insert: few evictions
    ev = engine.FakeNetEvaluator(0)
    roots, _ = _roots(eng, n, 8, seed=1)
    hits = []
    snaps = []
    for rnd in range(3):
        if rnd == 2:
            eng.clear_eval_cache()
        eng.reset_roots(roots)
        eng.run_search(sims, ev, graph_waves=4, adaptive=True)
        info = eng.status()
        hits.append((info["cache_hits"] / info["sims"], (info["cache_hits"] + info["terminal_leaves"]) / info["sims"]))
        snaps.append(_snapshot(eng))
    _same(snaps[0], snaps[1], "warm")
    _same(snaps[0], snaps[2], "cleared")
    assert hits[1][1] > 0.97 > hits[0][1]  # (nearly: direct-mapped) every leaf of the repeat is terminal or a hit
    assert abs(hits[2][0] - hits[0][0]) < 0.05     # cleared: back to the within-search hit rate
    eng.close()


def test_cache_with_real_net_matches_uncached(mods):
    """SimpleNN (bf16, fused plan): the same leaves get the same evaluation whether the net computes them (in whatever
    batch row, at whatever batch size of the adaptive loop) or the table returns them."""
    engine, _ = mods
    from dotsboxesaz_b200.dots_boxes.dots_boxes_nn import SimpleNN
    from dotsboxesaz_b200.nn import FusedSimpleNN
    n, sims = 512, 160
    torch.manual_seed(0)
    model = SimpleNN(board=(3, 3))
    plain = engine.Engine((3, 3), n_games=n, max_nodes=sims + 16)
    roots, _ = _roots(plain, n, 10, seed=11)
    ev0 = FusedSimpleNN(model, plain)
    plain.reset_roots(roots)
    plain.run_search(sims, ev0, graph_waves=8)
    ref = _snapshot(plain)
    plain.close()
    eng = engine.Engine((3, 3), n_games=n, max_nodes=sims + 16, eval_cache=16)
    ev1 = FusedSimpleNN(model, eng)
    eng.reset_roots(roots)
    eng.run_search(sims, ev1, graph_waves=8, adaptive=True)
    got = _snapshot(eng)
    assert eng.status()["cache_hits"] > 0
    same = (ref["visits"] == got["visits"]).all(1).mean()
    # library GEMM/conv kernels may pick another tiling at another batch size; rows must still agree almost always
    assert same > 0.98, same
    eng.close()


@pytest.mark.parametrize("board", [(6, 6), (7, 7), (4, 7)])
def test_cache_on_large_boards(mods, board):
    """Boards with more than 88 actions (the key no longer fits 96 bits: cells carry alternating slices of the 136-bit key):
    cached == uncached bit for bit, and the table is used."""
    engine, oracle = mods
    ev = engine.FakeNetEvaluator(0)
    n, sims = 48, 150
    plain = engine.Engine(board, n_games=n, max_nodes=4 * sims + 64)
    roots, played = _roots(plain, n, 30, seed=11)
    ref = _play(plain, ev, roots, sims, 3, noise_seed=5)
    plain.close()
    eng = engine.Engine(board, n_games=n, max_nodes=4 * sims + 64, eval_cache=12)
    got = _play(eng, ev, roots.clone(), sims, 3, noise_seed=5, graph_waves=4, adaptive=True)
    for m, (a, b) in enumerate(zip(ref, got)):
        _same(a, b, (board, "move", m))
    assert eng.status()["cache_hits"] > 0
    eng.close()
