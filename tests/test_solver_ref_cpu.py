"""CPU: the two references of the exact solver (oracle/solver_ref.py) against the rules and against each other.
The integer rules of the minimax search follow oracle/py_port.Board move for move; the sign of d + v(M) from the NumPy
retrograde table equals the minimax outcome on every reachable (edges, score) state of the small boards, and equals
get_result() on every terminal one."""
import numpy as np
import pytest

from oracle import py_port as pp
from oracle import solver_ref


@pytest.mark.parametrize("board", [(1, 1), (1, 4), (2, 3), (3, 3), (3, 4), (2, 6), (4, 1)])
def test_integer_rules_match_py_port(board):
    L, C = board
    mini = solver_ref.MinimaxOutcome(L, C)
    rng = np.random.RandomState(L * 10 + C)
    pp.Board.configure(L, C)
    try:
        for _ in range(30):
            b = pp.Board()
            edges, btc2, tp = mini.initial()
            while True:
                assert tp == b.to_play
                assert btc2 == (int(2 * b.need[0]), int(2 * b.need[1]))
                assert solver_ref.result(btc2, tp) == b.result()
                assert sum(1 << a for a in b.legal(as_indices=True)) == mini.g.real_mask & ~edges
                if b.result() is not None:
                    break
                a = int(rng.choice(b.legal(as_indices=True)))
                done = b.apply(a)
                edges, btc2, tp, n = mini.play(edges, btc2, tp, a)
                assert n == len(done)
    finally:
        pp.Board.configure(3, 3)


@pytest.mark.parametrize("board", [(1, 1), (1, 2), (1, 3), (1, 4), (2, 1), (2, 2), (2, 3), (3, 2)])
def test_retrograde_sign_equals_minimax(board):
    mini = solver_ref.MinimaxOutcome(*board)
    g = mini.g
    T = solver_ref.retrograde_numpy(*board)
    assert T.dtype == np.int8 and T.shape == (1 << g.E,) and not (T == -128).any()
    terminal = 0
    for edges, btc2, tp in mini.reachable():
        d, d2 = solver_ref.lead(g, edges, btc2, tp)
        assert d == d2
        o = int(np.sign(d + int(T[g.compact_mask(edges)])))
        assert o == mini.outcome(edges, btc2, tp), (edges, btc2, tp)
        r = solver_ref.result(btc2, tp)
        if r is not None:
            assert o == r
            terminal += 1
    assert terminal > 0


def test_1x1_value():
    """The fourth edge closes the only box, and the second player plays it."""
    assert int(solver_ref.retrograde_numpy(1, 1)[0]) == -1
