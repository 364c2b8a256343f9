"""Exact endgame play on every board the engine supports (A <= 128 actions: 4x4, 5x5, 6x6, 7x7, 1x31, ...).

A position with f free edges is solved by a retrograde over the 2^f subsets of those edges, in shared memory
(csrc/dbaz_endgame.cuh and DESIGN.md §11 give the definitions).  It is solvable when f <= max_free <= 16; its final
margin, outcome and move margins are those of the 32-edge table of solver.py, which the two must agree on byte for byte.
No table is kept, and nothing needs solving up front.

EndgameSolver       per-state queries: margins, outcomes, move margins, optimal moves, which states are solvable.
DeepEndgameSolver   the same queries up to f <= 32 (DESIGN.md §13): positions with 17 <= f free edges are solved in a
                    2^f-byte table each in device memory, outside CUDA graphs.
EndgameEvaluator    wraps any evaluator: exact priors and values on the leaves that are solvable, the inner evaluator's
                    output on every other leaf.
solver.grade / solver.grade_samples take either endgame solver too and grade the solvable rows.
"""
import ctypes as C

import numpy as np
import torch

from ._capi import ENDGAME_DEEP_GEOM_BYTES, RESULT_NONE
from .engine import EngineError, _ptr
from .solver import ILLEGAL


class EndgameSolver:
    """Exact values of positions with at most `max_free` (0 .. 16) free edges, on the engine's board; every query runs on
    the engine's current stream.  Rows of unsolvable positions read ILLEGAL (-128) everywhere."""

    def __init__(self, engine, max_free=16):
        self.eng = engine
        self.max_free = int(max_free)
        self.L, self.C, self.A = engine.L, engine.C, engine.A
        self.E = self.L * (self.C + 1) + self.C * (self.L + 1)
        self.LC = self.L * self.C
        rows, cols = self.L + 1, self.C + 1
        plane = rows * cols
        real = [a for a in range(2 * plane) if (a < plane and a % cols < self.C) or (a >= plane and (a - plane) // cols < self.L)]
        words = [0, 0]
        for a in real:
            words[a >> 6] |= 1 << (a & 63)
        # as int64 tensors (bit 63 is the sign bit)
        self._real = torch.tensor([w - (1 << 64) if w >> 63 else w for w in words], dtype=torch.int64, device=engine.device)
        self._box_actions = torch.tensor([[l * cols + c, (l + 1) * cols + c, plane + l * cols + c, plane + l * cols + c + 1]
                                          for l in range(self.L) for c in range(self.C)], dtype=torch.int64, device=engine.device)

    def _ck(self, rc):
        if rc != 0:
            raise EngineError(self.eng.lib.dbaz_last_error(self.eng._h).decode())

    def moves(self, states):
        """(move margins int8 [n, A] with ILLEGAL for played edges and padding, final margins int8 [n]); every byte of an
        unsolvable row is ILLEGAL."""
        eng = self.eng
        states = eng._states_arg(states)
        n = states.shape[0]
        mm = torch.empty((n, self.A), dtype=torch.int8, device=eng.device)
        mg = torch.empty((n,), dtype=torch.int8, device=eng.device)
        self._ck(eng.lib.dbaz_endgame_moves(eng._h, _ptr(states), _ptr(mm), _ptr(mg), self.max_free, n, eng._stream()))
        return mm, mg

    def free_edges(self, states):
        """Number of free real edges f of every state, int64 [n]."""
        states = self.eng._states_arg(states)
        free = self._real.unsqueeze(0) & ~states[:, :2]
        bits = (free.unsqueeze(-1) >> torch.arange(64, device=states.device)) & 1
        return bits.sum((1, 2))

    def solvable(self, states):
        """bool [n]: f <= max_free."""
        return self.free_edges(states) <= self.max_free

    def margin(self, states):
        """Final margin d + v(M), int8 [n]; ILLEGAL for unsolvable states."""
        return self.moves(states)[1]

    def outcome(self, states):
        """sign(final margin), int8 [n]: 1 win, 0 draw, -1 loss for the player to move; ILLEGAL for unsolvable states."""
        mg = self.margin(states)
        return torch.where(mg == ILLEGAL, mg, torch.sign(mg))

    def move_margins(self, states):
        """Final margin after each legal action, seen by the player to move before it; ILLEGAL elsewhere.  int8 [n, A]."""
        return self.moves(states)[0]

    def optimal_moves(self, states, kind="outcome"):
        """bool [n, A]: legal moves that keep the outcome (kind="outcome") or the final margin (kind="margin"); no move
        of an unsolvable state."""
        mm, mg = self.moves(states)
        if kind == "outcome":
            return (mm != ILLEGAL) & (torch.sign(mm) == torch.sign(mg).unsqueeze(1))
        if kind == "margin":
            return (mm != ILLEGAL) & (mm == mg.unsqueeze(1))
        raise ValueError("kind must be 'outcome' or 'margin'")

    def evaluate(self, eng, leaf_states, priors, values, mode=0, keep_priors=False):
        """dbaz_endgame_eval on an engine of the same board: on the rows of solvable leaves, priors uniform over the
        outcome-optimal moves (untouched with keep_priors) and values the outcome (mode 0) or final margin / (L C)
        (mode 1); every other row is left as it is."""
        n = leaf_states.shape[0]
        eng._ck(eng.lib.dbaz_endgame_eval(eng._h, _ptr(leaf_states), _ptr(priors), _ptr(values), int(mode), 1 if keep_priors else 0,
                                          self.max_free, n, eng._stream()))

    def adjudicate(self, bufs, margin, first=False):
        """dbaz_selfplay_adjudicate, after Engine.selfplay_restart(bufs, first): every game of the asynchronous self-play
        loop whose new root has at most max_free free edges ends there, with the root's final margin in margin (int8
        [n_games], ILLEGAL elsewhere)."""
        eng = self.eng
        eng._ck(eng.lib.dbaz_selfplay_adjudicate(eng._h, C.byref(bufs), _ptr(margin), self.max_free, 1 if first else 0, eng._stream()))

    def play_out(self, bufs, exact_margin, kind="outcome", first=False):
        """dbaz_selfplay_exact_endgame, after Engine.selfplay_restart(bufs, first): every game of the asynchronous self-play
        loop whose new root has at most max_free free edges is played out from there with optimal moves (kind "outcome" or
        "margin"), one history row per ply with the optimal moves as its visits, and ends with the root's final margin in
        exact_margin (int8 [n_games], ILLEGAL elsewhere)."""
        eng = self.eng
        if kind not in ("outcome", "margin"):
            raise ValueError("kind must be 'outcome' or 'margin'")
        eng._ck(eng.lib.dbaz_selfplay_exact_endgame(eng._h, C.byref(bufs), _ptr(exact_margin), self.max_free,
                                                    0 if kind == "outcome" else 1, 1 if first else 0, eng._stream()))

    def full_states(self, n):
        """n states with every real edge played (f = 0)."""
        st = self.eng.new_states(n)
        st[:, :2] = self._real
        return st

    def states_from_planes(self, planes):
        """Packed states [n, 4] from feature rows (get_features().ravel(), int16 or uint8 as in SampleBatch.planes), on
        every board (both edge words).  The planes show the edges and btc2[to_play]; the other player's btc2 follows from
        the closed boxes (btc2[0] + btc2[1] = 2 LC - 2 closed).  The player to move is written as player 0, the move before
        as unknown."""
        eng = self.eng
        x = torch.as_tensor(planes).to(eng.device)
        R = x.shape[0]
        x = x.reshape(R, -1)
        P = (self.L + 1) * (self.C + 1)
        if x.shape[1] != 3 * P:
            raise ValueError("planes must have 3 * (L + 1) * (C + 1) = %d features per row" % (3 * P))
        bits = x[:, :2 * P].to(torch.int64) & 1
        k = x[:, 2 * P].to(torch.int64)
        if x.dtype == torch.uint8:  # int8(2 * boxes_to_close) stored as a byte
            k = torch.where(k > 127, k - 256, k)
        padded = torch.zeros((R, 128), dtype=torch.int64, device=eng.device)
        padded[:, :2 * P] = bits
        shifts = torch.arange(64, device=eng.device)
        closed = bits[:, self._box_actions].all(-1).sum(1)
        out = torch.zeros((R, 16), dtype=torch.int16, device=eng.device)
        words = out.view(torch.int64)
        words[:, 0] = (padded[:, :64] << shifts).sum(1)  # distinct bits: the sum is their OR, bit 63 included
        words[:, 1] = (padded[:, 64:] << shifts).sum(1)
        out[:, 8] = k.to(torch.int16)                                    # btc2[0]: the player to move
        out[:, 9] = (2 * self.LC - 2 * closed - k).to(torch.int16)       # btc2[1]
        out[:, 10] = -256                                                # to_play 0, just_played -1
        out[:, 12] = -1
        out[:, 13] = -1                                                  # parent -1
        out[:, 14] = -1                                                  # parent_action -1
        out[:, 15] = RESULT_NONE
        return words


SHALLOW_MAX_FREE = 16  # the shared-memory tier of EndgameSolver


class DeepEndgameSolver(EndgameSolver):
    """EndgameSolver up to `max_free` (17 .. 32) free edges.  Rows with f <= 16 are solved as by EndgameSolver(engine, 16),
    rows with 17 <= f <= max_free by dbaz_endgame_deep_moves (grouped by f, one 2^f-byte table per position in a
    workspace of `workspace_bytes`, allocated at the first deep query and kept; default: max(one position at max_free,
    1 GiB)), every other row reads ILLEGAL.  A position costs about f 2^(f-1) successor reads.
    Every query synchronises the host (it reads the rows' f and the solver's checks), so it cannot be captured in a CUDA
    graph: evaluate / adjudicate / play_out raise ValueError, and EndgameEvaluator does not take it."""

    def __init__(self, engine, max_free=24, workspace_bytes=None):
        max_free = int(max_free)
        if not SHALLOW_MAX_FREE < max_free <= 32:
            raise ValueError("max_free must be in [17, 32], got %d" % max_free)
        need = (1 << max_free) + ENDGAME_DEEP_GEOM_BYTES
        workspace_bytes = max(need, 1 << 30) if workspace_bytes is None else int(workspace_bytes)
        if workspace_bytes < need:
            raise ValueError("one position with %d free edges needs %d workspace bytes, got %d" % (max_free, need, workspace_bytes))
        super().__init__(engine, max_free)
        self.workspace_bytes = workspace_bytes
        self.workspace = None

    def moves(self, states):
        """(move margins int8 [n, A] with ILLEGAL for played edges and padding, final margins int8 [n]); every byte of a
        row with f > max_free is ILLEGAL.  Synchronises."""
        eng = self.eng
        states = eng._states_arg(states)
        n = states.shape[0]
        mm = torch.empty((n, self.A), dtype=torch.int8, device=eng.device)
        mg = torch.empty((n,), dtype=torch.int8, device=eng.device)
        self._ck(eng.lib.dbaz_endgame_moves(eng._h, _ptr(states), _ptr(mm), _ptr(mg), SHALLOW_MAX_FREE, n, eng._stream()))
        f = self.free_edges(states).cpu().numpy()
        for fv in np.unique(f[(f > SHALLOW_MAX_FREE) & (f <= self.max_free)]):
            idx = torch.from_numpy(np.flatnonzero(f == fv)).to(eng.device)
            sub = states[idx].contiguous()
            smm = torch.empty((sub.shape[0], self.A), dtype=torch.int8, device=eng.device)
            smg = torch.empty((sub.shape[0],), dtype=torch.int8, device=eng.device)
            if self.workspace is None:
                self.workspace = torch.empty((self.workspace_bytes,), dtype=torch.int8, device=eng.device)
            self._ck(eng.lib.dbaz_endgame_deep_moves(eng._h, _ptr(sub), sub.shape[0], int(fv), _ptr(self.workspace), self.workspace_bytes,
                                                     _ptr(smm), _ptr(smg), eng._stream()))
            mm[idx] = smm
            mg[idx] = smg
        return mm, mg

    def evaluate(self, *args, **kwargs):
        raise ValueError("DeepEndgameSolver synchronises the host and cannot run inside the search; use EndgameSolver (max_free <= 16)")

    def adjudicate(self, *args, **kwargs):
        raise ValueError("DeepEndgameSolver synchronises the host and cannot run inside self-play; use EndgameSolver (max_free <= 16)")

    play_out = adjudicate


class EndgameEvaluator:
    """`inner` (FakeNetEvaluator, an nn plan, SolverEvaluator, ...) followed by one k_endgame_eval over the same leaves:
    exact values on the leaves with at most endgame.max_free free edges, and exact priors there unless priors="inner".
    value="outcome": the leaf's outcome (+1 / 0 / -1); value="margin": final margin / (L C).  Works in every
    Engine.run_search mode and in BatchedSelfPlay, with the eval cache on: its output is a function of the cache key
    whenever the inner evaluator's is."""

    def __init__(self, inner, endgame, value="outcome", priors="exact"):
        if value not in ("outcome", "margin"):
            raise ValueError("value must be 'outcome' or 'margin'")
        if priors not in ("exact", "inner"):
            raise ValueError("priors must be 'exact' or 'inner'")
        if isinstance(endgame, DeepEndgameSolver):
            raise ValueError("the evaluator runs inside the search's CUDA graphs; DeepEndgameSolver cannot, use EndgameSolver")
        self.inner = inner
        self.endgame = endgame
        self.mode = 0 if value == "outcome" else 1
        self.keep_priors = priors == "inner"
        self.engine_launches = int(getattr(inner, "engine_launches", 0)) + 1  # the inner evaluator's kernels + k_endgame_eval
        q = getattr(inner, "batch_quantum", None)
        if q:
            self.batch_quantum = q  # the adaptive loop sizes its batches for the inner evaluator

    def __call__(self, eng):
        if (eng.L, eng.C) != (self.endgame.L, self.endgame.C):
            raise ValueError("the endgame solver is for a %dx%d board, the engine plays %dx%d" % (self.endgame.L, self.endgame.C, eng.L, eng.C))
        self.inner(eng)
        self.endgame.evaluate(eng, eng.leaf_states, eng.priors, eng.values, self.mode, self.keep_priors)
