"""CPU: the references of the endgame solver (tests/endgame_ref.py).  endgame_numpy's sub-table over a position's free
edges equals the full-game retrograde table on every superset of the played edges (small boards); on 4x4, 5x5 and 7x7
it equals margin_minimax, a negamax with plain rules over action-space masks, and its outcome has the sign of
MinimaxOutcome's."""
import numpy as np
import pytest

import endgame_ref
from oracle import solver_ref

SMALL = [(1, 1), (1, 2), (1, 3), (1, 4), (1, 5), (1, 6), (1, 7), (2, 1), (3, 1), (4, 1), (5, 1), (6, 1), (7, 1), (2, 2), (2, 3), (3, 2),
         (2, 4), (4, 2), (3, 3)]


def _random_edges(g, rng, n_free):
    """a random set of played edges leaving exactly n_free real edges free"""
    played = rng.permutation(len(g.real))[:g.E - n_free]
    return sum(1 << int(g.real[j]) for j in played)


def _random_scores(g, rng, edges):
    """(btc2, to_play) with the closed boxes split at random between the players"""
    closed = g.closed_boxes(edges)
    mine = int(rng.randint(0, closed + 1))
    return (g.LC - 2 * mine, g.LC - 2 * (closed - mine)), 0


@pytest.mark.parametrize("board", SMALL)
def test_subtable_equals_full_table(board):
    g = solver_ref.Geometry(*board)
    T = solver_ref.retrograde_numpy(*board)
    rng = np.random.RandomState(board[0] * 100 + board[1])
    for n_free in range(g.E + 1):
        for _ in range(3 if g.E > 16 else 6):
            edges = _random_edges(g, rng, n_free)
            sub = endgame_ref.endgame_numpy(g, edges)
            free = endgame_ref.free_edges(g, edges)
            assert sub.dtype == np.int8 and sub.shape == (1 << n_free,) and len(free) == n_free
            # local mask m -> compact mask of M | m
            M = g.compact_mask(edges)
            comp = np.array([1 << g.compact[a] for a in free], dtype=np.int64)
            m = np.arange(1 << n_free, dtype=np.int64)
            full = np.full(m.shape, M, dtype=np.int64)
            for i in range(n_free):
                full |= np.where((m >> i) & 1, comp[i], 0)
            assert np.array_equal(sub, T[full]), (board, edges)


@pytest.mark.parametrize("board", [(4, 4), (5, 5), (7, 7)])
def test_subtable_equals_margin_minimax(board):
    g = solver_ref.Geometry(*board)
    rng = np.random.RandomState(board[0] * 7 + board[1])
    mini = solver_ref.MinimaxOutcome(*board)
    memo = {}
    for n_free in range(11):
        for _ in range(4):
            edges = _random_edges(g, rng, n_free)
            sub = endgame_ref.endgame_numpy(g, edges)
            v = endgame_ref.margin_minimax(g, edges, memo)
            assert int(sub[0]) == v, (board, edges)
            # a few deeper entries: the sub-table at local mask m is the value after the free edges of m are played
            free = endgame_ref.free_edges(g, edges)
            for m in rng.randint(0, 1 << n_free, size=4):
                e2 = edges | sum(1 << a for i, a in enumerate(free) if (int(m) >> i) & 1)
                assert int(sub[int(m)]) == endgame_ref.margin_minimax(g, e2, memo)
            btc2, tp = _random_scores(g, rng, edges)
            d = solver_ref.lead(g, edges, btc2, tp)
            assert d[0] == d[1]
            assert int(np.sign(d[0] + v)) == mini.outcome(edges, btc2, tp), (board, edges, btc2)
            mm, final = endgame_ref.endgame_moves(g, edges, btc2, tp, sub)
            assert final == d[0] + v
            assert sorted(np.flatnonzero(mm != -128).tolist()) == free


def test_margin_minimax_terminal_and_last_edge():
    g = solver_ref.Geometry(1, 1)
    assert endgame_ref.margin_minimax(g, g.real_mask) == 0
    # three edges played: the last one closes the box for the player to move
    assert endgame_ref.margin_minimax(g, g.real_mask & ~(1 << g.real[0])) == 1
    assert endgame_ref.margin_minimax(g, 0) == int(solver_ref.retrograde_numpy(1, 1)[0]) == -1
