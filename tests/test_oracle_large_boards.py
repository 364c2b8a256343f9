"""Pins the C oracle (oracle/dbaz_oracle.c) against the independent Python port (oracle/py_port.py) on boards past
5x5 -- up to A = 128 actions, the engine's limit -- where no fixture recorded from the reference exists.  The GPU
tests of these boards (test_gpu_large_boards.py) take the oracle as their reference; this file is what that reference
stands on.  CPU only.

Only searches with one simulation in flight (max_pending = 1) are compared.  With K > 1 the port is not a reference:
its fake net never suspends (an `async def` without an await), so every simulation it starts runs to its backup before
the next one descends, and its virtual losses never overlap the way the reference's do with a batching proxy in front
of the net.  The oracle models the overlapping schedule; for K > 1 it is pinned by the mcts_pending fixtures (boards up
to 5x5) alone."""
import asyncio
import warnings

import numpy as np
import pytest

from oracle import oracle
from oracle import py_port as pp

# A = 2 (L+1)(C+1): 98, 128, 80, 80, 112, 32, 128, 128, 128, 8
BOARDS = [(6, 6), (7, 7), (4, 7), (7, 4), (6, 7), (1, 7), (1, 31), (31, 1), (3, 15), (1, 1)]


def _nn(kind):
    async def nn(board):
        return pp.fake_nn_eval(board, kind)
    return nn


@pytest.mark.parametrize("board", BOARDS)
def test_rules_match_py_port(board):
    """Whole random games, every ply: board bytes, to_play, just_played, 2 * boxes_to_close, the full-width hash
    (sum of 1 << move over every move: 128 bits on 7x7), the second hash word, features, result and the closed boxes."""
    L, C = board
    pp.Board.configure(L, C)
    rng = np.random.RandomState(L * 100 + C)
    for game in range(10):
        og, b = oracle.OracleGame(L, C), pp.Board()
        assert og.A == b.n_actions
        plies = 0
        while og.result() is None:
            legal = np.flatnonzero(og.valid_moves())
            assert legal.tolist() == b.legal(as_indices=True), (board, game, plies)
            mv = int(rng.choice(legal))
            closed = og.play_(mv)
            assert [list(x) for x in closed] == [list(x) for x in b.apply(mv)], (board, game, plies, mv)
            plies += 1
            rec = og.record()
            where = (board, game, plies, mv)
            assert rec["board"] == bytes(b.cells.ravel().tolist()).hex(), where
            assert (rec["to_play"], rec["just_played"]) == (b.to_play, b.just_played), where
            assert rec["btc2"] == [int(round(2 * x)) for x in b.need], where
            assert int(rec["hash0"]) == int(b.key[0]), where
            assert rec["hash1_x2"] == int(round(2 * b.key[1])), where
            assert np.array_equal(og.features().ravel().astype(np.int8), b.planes().ravel().astype(np.int8)), where
            assert rec["result"] == (2 if b.result() is None else b.result()), where
        n_edges = L * (C + 1) + C * (L + 1)
        assert og.result() is not None and plies <= n_edges
        # a played edge, a padding cell (the last action), A and -1 are illegal
        for bad in (mv, og.A - 1, og.A, -1):
            with pytest.raises(ValueError):
                og.copy().play_(bad)
        with pytest.raises(ValueError):
            pp.Board(b).apply(og.A - 1)


@pytest.mark.parametrize("kind", [0, 1])
@pytest.mark.parametrize("board", BOARDS)
def test_sequential_search_matches_py_port(board, kind):
    """Three 300-simulation searches (one simulation in flight), Dirichlet noise in the first, each followed by a re-root:
    reuse onto the most visited child, reuse onto an unvisited legal child, a fresh tree.  Visit counts, W, priors, the
    root's N and the tree statistics must be equal after every search and every re-root."""
    warnings.filterwarnings("ignore")
    L, C = board
    pp.Board.configure(L, C)
    rng = np.random.RandomState(7 * L + C + kind)
    og, b = oracle.OracleGame(L, C), pp.Board()
    n_edges = L * (C + 1) + C * (L + 1)
    for _ in range(min(5, n_edges - 3)):
        mv = int(rng.choice(np.flatnonzero(og.valid_moves())))
        og.play_(mv)
        b.apply(mv)
    tree, root = oracle.OracleTree(L, C, og.s, kind=kind), pp.new_root(b)

    def check(where):
        r = tree.root()
        assert r["visits"].tolist() == root.child_N.tolist(), where
        assert np.array_equal(r["W"], root.child_W), where
        assert np.array_equal(r["priors"], np.asarray(root.prior, dtype=np.float64)), where
        assert r["root_N"] == int(root.N_own), where
        stats = root.parent.stats()
        assert r["stats"][:3] == [int(x) for x in stats[:3]], (where, r["stats"], stats)
        assert np.float32(r["stats"][3]) == np.float32(stats[3]), where
        return r

    reads, searched = 300, 0
    for step in range(3):
        if tree.root()["is_terminal"]:
            break
        if step == 0:
            seed = 1000 + L * 40 + C
            np.random.seed(seed)
            asyncio.run(pp.uct_search(root, reads, _nn(kind), max_pending=1, dirichlet=(0.8, 0.25)))
            valid = tree.root()["state"].valid_moves()
            noise = np.random.RandomState(seed).dirichlet(np.ones(tree.A) * 0.8, 1).ravel() * valid
            tree.search(reads, noise=noise, coeff=0.25)
        else:
            asyncio.run(pp.uct_search(root, reads, _nn(kind), max_pending=1))
            tree.search(reads)
        r = check((board, kind, step, "search"))
        searched += 1
        legal = np.flatnonzero(r["state"].valid_moves())
        unvisited = [int(a) for a in legal if r["visits"][a] == 0]
        mv = unvisited[0] if step == 1 and unvisited else int(np.argmax(r["visits"]))
        tree.reroot(mv, step < 2)
        root = pp.reroot(root, mv, step < 2)
        check((board, kind, step, "reroot", mv))
    assert searched >= 2
