"""CPU references for the exact solver (dotsboxesaz_b200/csrc/dbaz_solver.cuh) -- TEST INFRASTRUCTURE ONLY.

Two independent computations of what the GPU table encodes:
  MinimaxOutcome    a memoised game-outcome search that stops at a majority, as the reference's get_result() does,
                    written with plain integer rules over the action-space edge mask (no compact indices, no margins);
  retrograde_numpy  the full-game margin table v(M) over compact masks, one NumPy pass per popcount layer.
The two agree through sign(d + v(M)) == outcome (tests/test_solver_ref_cpu.py); the GPU table is compared with the second.
"""
import numpy as np


class Geometry:
    """Actions, real edges and boxes of an L x C board, restated from dots_boxes_game.py's layout: action a = p * plane +
    l * (C + 1) + c, p = 0 horizontal edges (padding column c == C), p = 1 vertical edges (padding row l == L)."""

    def __init__(self, L, C):
        self.L, self.C = L, C
        self.rows, self.cols = L + 1, C + 1
        self.plane = self.rows * self.cols
        self.A = 2 * self.plane
        self.real = [a for a in range(self.A) if (a < self.plane and a % self.cols < C) or (a >= self.plane and (a - self.plane) // self.cols < L)]
        self.E = len(self.real)
        self.LC = L * C
        self.compact = {a: j for j, a in enumerate(self.real)}
        # the four edges of box (l, c) (dots_boxes_game.py:102-104), box index l * C + c
        self.box_actions = [(l * self.cols + c, (l + 1) * self.cols + c, self.plane + l * self.cols + c, self.plane + l * self.cols + c + 1)
                            for l in range(L) for c in range(C)]
        self.box_mask = [sum(1 << a for a in b) for b in self.box_actions]
        self.box_cmask = [sum(1 << self.compact[a] for a in b) for b in self.box_actions]
        # boxes an action borders, in the order play_ tests them (dots_boxes_game.py:72-79)
        self.boxes_of = {}
        for a in self.real:
            p, rem = divmod(a, self.plane)
            l, c = divmod(rem, self.cols)
            if p == 0:
                cand = ([(l - 1, c)] if l > 0 else []) + ([(l, c)] if l < L else [])
            else:
                cand = ([(l, c - 1)] if c > 0 else []) + ([(l, c)] if c < C else [])
            self.boxes_of[a] = [bl * C + bc for bl, bc in cand]
        self.real_mask = sum(1 << a for a in self.real)

    def compact_mask(self, edges):
        return sum(1 << j for j, a in enumerate(self.real) if (edges >> a) & 1)

    def closed_boxes(self, edges):
        return sum(1 for m in self.box_mask if edges & m == m)


def result(btc2, to_play):
    """get_result() (dots_boxes_game.py:51-59) on doubled boxes-to-close: 1 / -1 / 0 seen by the player to move, None."""
    mine, other = btc2[to_play], btc2[1 - to_play]
    if mine == 0 and other == 0:
        return 0
    if mine < 0:
        return 1
    if other < 0:
        return -1
    return None


class MinimaxOutcome:
    """Game outcome under best play, seen by the player to move, by memoised search over (edges, mine2, other2)."""

    def __init__(self, L, C):
        self.g = Geometry(L, C)
        self.memo = {}

    def initial(self):
        """(edges, btc2, to_play) of the empty board."""
        return 0, (self.g.LC, self.g.LC), 0

    def play(self, edges, btc2, to_play, a):
        """play_ (dots_boxes_game.py:61-89) with integers: returns (edges, btc2, to_play, boxes closed)."""
        if not (self.g.real_mask >> a) & 1 or (edges >> a) & 1:
            raise ValueError("Illegal move: %s" % a)
        edges |= 1 << a
        n = sum(1 for b in self.g.boxes_of[a] if edges & self.g.box_mask[b] == self.g.box_mask[b])
        if n:
            btc2 = (btc2[0] - 2 * n, btc2[1]) if to_play == 0 else (btc2[0], btc2[1] - 2 * n)
        else:
            to_play = 1 - to_play
        return edges, btc2, to_play, n

    def outcome(self, edges, btc2, to_play):
        return self._outcome(edges, btc2[to_play], btc2[1 - to_play])

    def _outcome(self, edges, mine, other):
        r = result((mine, other), 0)
        if r is not None:
            return r
        key = (edges, mine, other)
        got = self.memo.get(key)
        if got is not None:
            return got
        best = -2
        free = self.g.real_mask & ~edges
        while free and best < 1:
            low = free & -free
            free ^= low
            e2 = edges | low
            a = low.bit_length() - 1
            n = sum(1 for b in self.g.boxes_of[a] if e2 & self.g.box_mask[b] == self.g.box_mask[b])
            v = self._outcome(e2, mine - 2 * n, other) if n else -self._outcome(e2, other, mine)
            best = max(best, v)
        self.memo[key] = best
        return best

    def reachable(self):
        """Every (edges, btc2, to_play) reachable from the empty board under the reference's rules (a game stops at a
        result), terminal states included."""
        start = self.initial()
        seen = {start}
        stack = [start]
        while stack:
            edges, btc2, tp = stack.pop()
            if result(btc2, tp) is not None:
                continue
            free = self.g.real_mask & ~edges
            while free:
                low = free & -free
                free ^= low
                e2, b2, t2, _ = self.play(edges, btc2, tp, low.bit_length() - 1)
                s = (e2, b2, t2)
                if s not in seen:
                    seen.add(s)
                    stack.append(s)
        return seen


def _popcount32(x):
    x = x - ((x >> 1) & 0x55555555)
    x = (x & 0x33333333) + ((x >> 2) & 0x33333333)
    x = (x + (x >> 4)) & 0x0F0F0F0F
    return (x * 0x01010101 & 0xFFFFFFFF) >> 24


def retrograde_numpy(L, C):
    """int8[2^E]: v(M) for every compact mask M, v(full) = 0, v(M) = max over free j of (c_j ? c_j + v(M|j) : -v(M|j))."""
    g = Geometry(L, C)
    E = g.E
    ebox = [[g.box_cmask[b] for b in g.boxes_of[a]] for a in g.real]
    N = 1 << E
    T = np.full(N, -128, dtype=np.int8)
    T[N - 1] = 0
    pop = _popcount32(np.arange(N, dtype=np.int64))
    order = np.argsort(pop, kind="stable")
    bounds = np.concatenate([[0], np.cumsum(np.bincount(pop, minlength=E + 1))])
    for k in range(E - 1, -1, -1):
        layer = order[bounds[k]:bounds[k + 1]]
        best = np.full(layer.shape, -128, dtype=np.int16)
        for j in range(E):
            bit = 1 << j
            free = (layer & bit) == 0
            s = layer | bit
            v = T[s].astype(np.int16)
            c = np.zeros(layer.shape, dtype=np.int16)
            for bm in ebox[j]:
                c += (s & bm) == bm
            best = np.where(free, np.maximum(best, np.where(c > 0, c + v, -v)), best)
        T[layer] = best.astype(np.int8)
    return T


def lead(g, edges, btc2, to_play):
    """The mover's score lead d two ways: (btc2[other] - btc2[mine]) / 2 and LC - btc2[mine] - closed boxes."""
    return (btc2[1 - to_play] - btc2[to_play]) // 2, g.LC - btc2[to_play] - g.closed_boxes(edges)


def move_margins(g, T, edges, btc2, to_play):
    """{action: move margin} of every legal action, from the table T (host recount of dbaz_solver_moves)."""
    d = lead(g, edges, btc2, to_play)[1]
    M = g.compact_mask(edges)
    out = {}
    for a in g.real:
        if (edges >> a) & 1:
            continue
        e2 = edges | (1 << a)
        n = sum(1 for b in g.boxes_of[a] if e2 & g.box_mask[b] == g.box_mask[b])
        v = int(T[M | (1 << g.compact[a])])
        out[a] = d + (n + v if n else -v)
    return out
