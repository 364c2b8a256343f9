"""CPU references for the endgame solver (dotsboxesaz_b200/csrc/dbaz_endgame.cuh) -- TEST INFRASTRUCTURE ONLY.

Built on the geometry and lead of oracle/solver_ref.py:
  endgame_numpy   the sub-table v_s(m) over a position's free edges, one NumPy pass per popcount layer, as
                  retrograde_numpy does for the full game;
  endgame_moves   move margins and final margin of a position from that sub-table;
  margin_minimax  a memoised margin negamax with plain rules over action-space edge masks (no local or compact indices),
                  for positions with few free edges on any board.
"""
import numpy as np

from oracle.solver_ref import _popcount32, lead


def free_edges(g, edges):
    """The free real edges of a position in increasing action order: local edge i is the i-th of them."""
    return [a for a in g.real if not (edges >> a) & 1]


def endgame_numpy(g, edges):
    """int8[2^f]: the endgame sub-table v_s(m) over the f free edges of the position with played edges `edges` (action
    space), m a local mask.  A box closes when every one of its free edges is in m; v_s(F) = 0, v_s(m) = max over free i
    of (c_i ? c_i + v_s(m|i) : -v_s(m|i)).  So entry 0 is v(M) of the full-game table."""
    free = free_edges(g, edges)
    f = len(free)
    local = {a: i for i, a in enumerate(free)}
    ebox = [[sum(1 << local[e] for e in g.box_actions[b] if e in local) for b in g.boxes_of[a]] for a in free]
    N = 1 << f
    T = np.full(N, -128, dtype=np.int8)
    T[N - 1] = 0
    pop = _popcount32(np.arange(N, dtype=np.int64))
    order = np.argsort(pop, kind="stable")
    bounds = np.concatenate([[0], np.cumsum(np.bincount(pop, minlength=f + 1))])
    for k in range(f - 1, -1, -1):
        layer = order[bounds[k]:bounds[k + 1]]
        best = np.full(layer.shape, -128, dtype=np.int16)
        for i in range(f):
            bit = 1 << i
            is_free = (layer & bit) == 0
            s = layer | bit
            v = T[s].astype(np.int16)
            c = np.zeros(layer.shape, dtype=np.int16)
            for bm in ebox[i]:
                c += (s & bm) == bm
            best = np.where(is_free, np.maximum(best, np.where(c > 0, c + v, -v)), best)
        T[layer] = best.astype(np.int8)
    return T


def endgame_moves(g, edges, btc2, to_play, T=None):
    """(move margins int [A] with -128 for played edges and padding, final margin) of a position from its endgame
    sub-table (host recount of dbaz_endgame_moves for a solvable position)."""
    T = endgame_numpy(g, edges) if T is None else T
    d = lead(g, edges, btc2, to_play)[1]
    free = free_edges(g, edges)
    mm = np.full(g.A, -128, dtype=np.int64)
    for i, a in enumerate(free):
        e2 = edges | (1 << a)
        n = sum(1 for b in g.boxes_of[a] if e2 & g.box_mask[b] == g.box_mask[b])
        v = int(T[1 << i])
        mm[a] = d + (n + v if n else -v)
    return mm, d + int(T[0])


def margin_minimax(g, edges, memo=None):
    """v(M) by memoised negamax with plain rules over action-space edge masks (no local or compact indices): the largest
    net number of boxes the player to move can still gain from the position with played edges `edges`, playing to the
    end.  Meant for positions with few free edges, on any board."""
    memo = {} if memo is None else memo
    got = memo.get(edges)
    if got is not None:
        return got
    free = g.real_mask & ~edges
    best = 0 if not free else -10 ** 6
    while free:
        low = free & -free
        free ^= low
        a = low.bit_length() - 1
        e2 = edges | low
        n = sum(1 for b in g.boxes_of[a] if e2 & g.box_mask[b] == g.box_mask[b])
        v = margin_minimax(g, e2, memo)
        best = max(best, n + v if n else -v)
    memo[edges] = best
    return best
