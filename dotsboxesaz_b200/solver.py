"""Exact play on boards of at most 32 real edges (1x1..1x10, 2x2..2x6, 3x3, 3x4 and their transposes).

A retrograde table holds, for every set M of played edges, v(M): the largest net number of boxes the player to move can
still gain against best play (csrc/dbaz_solver.cuh and DESIGN.md §10 give the definitions).  With the mover's lead
d = LC - btc2[to_play] - closed(M), a position's final margin is d + v(M) and its outcome sign(d + v(M)), seen by the
player to move as get_result() sees it.  3x3 takes 16 MiB, 3x4 2 GiB, 2x6 4 GiB of device memory.

Solver            the table and per-state queries: margins, outcomes, move margins, optimal moves.
SolverEvaluator   a perfect evaluator for Engine.run_search (drop-in for engine.FakeNetEvaluator).
grade             policy / value / z figures of a batch of positions against perfect play; grade_samples for a SampleBatch.
play_vs_solver    games of a model (search + evaluator) against the perfect opponent, with blunder counts.
"""
import numpy as np
import torch

from ._capi import RESULT_NONE
from .engine import EngineError, _ptr
from .self_play import _n_searches

ILLEGAL = -128  # move margin of a played edge or padding slot


class Solver:
    """The exact table of the engine's board.  solve() fills it; every query runs on the engine's current stream."""

    def __init__(self, engine):
        self.eng = engine
        self.L, self.C, self.A = engine.L, engine.C, engine.A
        self.E = self.L * (self.C + 1) + self.C * (self.L + 1)
        self.LC = self.L * self.C
        self.table = None
        rows, cols = self.L + 1, self.C + 1
        plane = rows * cols
        # the four actions of every box (dots_boxes_game.py:102-104), for states_from_planes
        self._box_actions = torch.tensor([[l * cols + c, (l + 1) * cols + c, plane + l * cols + c, plane + l * cols + c + 1]
                                          for l in range(self.L) for c in range(self.C)], dtype=torch.int64, device=engine.device)

    def _ck(self, rc):
        if rc != 0:
            raise EngineError(self.eng.lib.dbaz_last_error(self.eng._h).decode())

    def solve(self, table=None):
        """Fill `table` (int8, 2^E bytes on the engine's device; allocated when None) and keep it as self.table.
        Raises EngineError for boards with more than 32 edges or a table of the wrong size.  Synchronises."""
        eng = self.eng
        if table is None and self.E <= 32:
            table = torch.empty((1 << self.E,), dtype=torch.int8, device=eng.device)
        nbytes = 0 if table is None else table.numel() * table.element_size()
        self._ck(eng.lib.dbaz_solver_solve(eng._h, _ptr(table), nbytes, eng._stream()))
        self.table = table
        return self

    def _need_table(self):
        if self.table is None:
            raise RuntimeError("Solver.solve() has not been called")
        return self.table

    def moves(self, states):
        """(move margins int8 [n, A] with ILLEGAL for played edges and padding, final margins int8 [n])."""
        eng = self.eng
        table = self._need_table()
        states = eng._states_arg(states)
        n = states.shape[0]
        mm = torch.empty((n, self.A), dtype=torch.int8, device=eng.device)
        mg = torch.empty((n,), dtype=torch.int8, device=eng.device)
        self._ck(eng.lib.dbaz_solver_moves(eng._h, _ptr(table), _ptr(states), _ptr(mm), _ptr(mg), n, eng._stream()))
        return mm, mg

    def margin(self, states):
        """Final margin d + v(M), int8 [n]: boxes the player to move ends ahead by under best play."""
        return self.moves(states)[1]

    def outcome(self, states):
        """sign(final margin), int8 [n]: 1 win, 0 draw, -1 loss for the player to move."""
        return torch.sign(self.margin(states))

    def move_margins(self, states):
        """Final margin after each legal action, seen by the player to move before it; ILLEGAL elsewhere.  int8 [n, A]."""
        return self.moves(states)[0]

    def optimal_moves(self, states, kind="outcome"):
        """bool [n, A]: legal moves that keep the outcome (kind="outcome") or the final margin (kind="margin")."""
        mm, mg = self.moves(states)
        if kind == "outcome":
            return (mm != ILLEGAL) & (torch.sign(mm) == torch.sign(mg).unsqueeze(1))
        if kind == "margin":
            return (mm != ILLEGAL) & (mm == mg.unsqueeze(1))
        raise ValueError("kind must be 'outcome' or 'margin'")

    def evaluate(self, eng, leaf_states, priors, values, mode=0):
        """dbaz_solver_eval on an engine of the same board: priors uniform over the outcome-optimal moves, values the
        outcome (mode 0) or final margin / (L C) (mode 1)."""
        n = leaf_states.shape[0]
        eng._ck(eng.lib.dbaz_solver_eval(eng._h, _ptr(self._need_table()), _ptr(leaf_states), _ptr(priors), _ptr(values), int(mode), n,
                                         eng._stream()))

    def states_from_planes(self, planes):
        """Packed states [n, 4] from feature rows (get_features().ravel(), int16 or uint8 as in SampleBatch.planes).  The
        planes show the edges and btc2[to_play]; the other player's btc2 follows from the closed boxes
        (btc2[0] + btc2[1] = 2 LC - 2 closed).  The player to move is written as player 0, the move before as unknown."""
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
        edges = (bits << torch.arange(2 * P, device=eng.device)).sum(1)  # every supported board has 2P <= 44 actions
        closed = bits[:, self._box_actions].all(-1).sum(1)
        out = torch.zeros((R, 16), dtype=torch.int16, device=eng.device)
        words = out.view(torch.int64)
        words[:, 0] = edges
        out[:, 8] = k.to(torch.int16)                                    # btc2[0]: the player to move
        out[:, 9] = (2 * self.LC - 2 * closed - k).to(torch.int16)       # btc2[1]
        out[:, 10] = -256                                                # to_play 0, just_played -1
        out[:, 12] = -1
        out[:, 13] = -1                                                  # parent -1
        out[:, 14] = -1                                                  # parent_action -1
        out[:, 15] = RESULT_NONE
        return words


class SolverEvaluator:
    """Perfect-play evaluator: drop-in for engine.FakeNetEvaluator in every Engine.run_search mode and in
    BatchedSelfPlay.  Its output is a function of the eval-cache key, so it can run with the cache on.
    value="outcome": the leaf's outcome (+1 / 0 / -1); value="margin": final margin / (L C)."""

    engine_launches = 1  # one k_solver_eval per wave

    def __init__(self, solver, value="outcome"):
        if value not in ("outcome", "margin"):
            raise ValueError("value must be 'outcome' or 'margin'")
        solver._need_table()
        self.solver = solver
        self.mode = 0 if value == "outcome" else 1

    def __call__(self, eng):
        if (eng.L, eng.C) != (self.solver.L, self.solver.C):
            raise ValueError("the solver's table is for a %dx%d board, the engine plays %dx%d" % (self.solver.L, self.solver.C, eng.L, eng.C))
        self.solver.evaluate(eng, eng.leaf_states, eng.priors, eng.values, self.mode)


def grade(solver, states, policy=None, value=None, z=None):
    """Figures of positions against perfect play (float64 means over the n rows):
    optimal_move_rate       share of rows whose policy argmax (lowest index on ties) is outcome-optimal
    optimal_mass            mean policy mass on outcome-optimal moves
    value_outcome_accuracy  share of rows where value > 1/3 (win), < -1/3 (loss) or else (draw) matches the outcome
    value_mse               mean squared error of value against the outcome
    z_agreement             share of rows whose sign(z) equals the outcome
    Only the figures whose inputs are given are returned, plus n.
    With an endgame.EndgameSolver the means run over the solvable rows only, and n_solved counts them."""
    mm, mg = solver.moves(states)
    dev = mm.device
    out = {"n": int(mm.shape[0])}
    keep = None
    if hasattr(solver, "max_free"):  # an EndgameSolver: unsolvable rows read ILLEGAL and are dropped
        keep = mg != ILLEGAL
        mm, mg = mm[keep], mg[keep]
        out["n_solved"] = int(mm.shape[0])
    o = torch.sign(mg).to(torch.float64)
    opt = (mm != ILLEGAL) & (torch.sign(mm) == torch.sign(mg).unsqueeze(1))
    if policy is not None:
        p = torch.as_tensor(policy).to(device=dev, dtype=torch.float64)
        p = (p.reshape(-1, solver.A)[keep] if keep is not None else p).reshape(mm.shape)
        best = p.max(1, keepdim=True).values
        ar = torch.arange(solver.A, device=dev)
        first = torch.where(p == best, ar, solver.A).min(1).values
        out["optimal_move_rate"] = opt.gather(1, first.unsqueeze(1)).double().mean().item()
        out["optimal_mass"] = (p * opt).sum(1).mean().item()
    if value is not None:
        v = torch.as_tensor(value).to(device=dev, dtype=torch.float64).reshape(-1)
        v = v[keep] if keep is not None else v
        pred = torch.where(v > 1.0 / 3.0, 1.0, torch.where(v < -1.0 / 3.0, -1.0, 0.0))
        out["value_outcome_accuracy"] = (pred == o).double().mean().item()
        out["value_mse"] = ((v - o) ** 2).mean().item()
    if z is not None:
        zz = torch.as_tensor(z).to(device=dev, dtype=torch.float64).reshape(-1)
        zz = zz[keep] if keep is not None else zz
        out["z_agreement"] = (torch.sign(zz) == o).double().mean().item()
    return out


def grade_samples(solver, batch):
    """grade() of a samples.SampleBatch: its positions rebuilt from the feature planes, pi as the policy, and z.  `solver`
    is a Solver or an endgame.EndgameSolver."""
    return grade(solver, solver.states_from_planes(batch.planes), policy=batch.pi, z=batch.z)


def play_vs_solver(engine, evaluator, params, solver, n_games, seed=0, start_states=None):
    """`n_games` lock-step games of a model against the perfect opponent, in the style of self_play.compute_elo: the
    model plays player 0 in even games and player 1 in odd ones; its moves come from Engine.run_search with
    params.self_play (budget, PUCT constants, Dirichlet noise, temperature schedule, tree reuse), on trees where the
    solver is to move the search is idle; the solver plays a uniformly random margin-optimal move.  Both sides' draws
    come from one device generator seeded with `seed`.
    start_states (int64 [n_games, 4], optional): the games start there instead of the empty board; move numbers (the
    temperature schedule) count from there.  With an endgame solver every start state must be solvable.  Each model
    search gets _n_searches(legal moves of its root) simulations.
    Returns dict(wins, draws, losses, model_moves, blunders) -- a blunder is a model move whose margin has a lower sign
    than the outcome of the position it was played from -- plus, on the device: result int8 [n_games] (the model's
    result), states [plies, n_games, 4], moves int32 [plies, n_games] (-1 once a game is over) and model bool
    [plies, n_games] (the model made that move)."""
    eng = engine
    n = eng.n_games
    if not 1 <= n_games <= n:
        raise ValueError("n_games must be in [1, engine.n_games]")
    if (eng.L, eng.C) != (solver.L, solver.C):
        raise ValueError("the solver and the engine play different boards")
    sp = params.self_play
    dev = eng.device
    num_read = sp.mcts.mcts_num_read
    alpha, coeff = sp.noise
    roots0 = None
    if start_states is not None:
        start_states = eng._states_arg(start_states)
        if start_states.shape[0] != n_games:
            raise ValueError("start_states must have n_games rows")
        if hasattr(solver, "max_free") and not bool(solver.solvable(start_states).all()):
            raise ValueError("every start state must have at most max_free = %d free edges" % solver.max_free)
        roots0 = eng.new_states(n)
        roots0[:n_games] = start_states
    eng.set_cpuct(sp.mcts.mcts_cpuct)
    eng.reset_roots(roots0)
    slot = torch.arange(n, device=dev)
    playing = slot < n_games
    model_player = slot % 2
    gen = torch.Generator(device=dev)
    gen.manual_seed(int(seed))
    temperature = None
    hist_states, hist_moves, hist_model = [], [], []
    model_moves = torch.zeros((), dtype=torch.int64, device=dev)
    blunders = torch.zeros((), dtype=torch.int64, device=dev)
    for move_i in range(solver.E):
        if move_i in sp.mcts.temperature:
            temperature = float(sp.mcts.temperature[move_i])
        roots = eng.root_states()
        active = (eng.result(roots) == RESULT_NONE) & playing
        if not bool(active.any()):
            break
        to_play = roots.view(torch.uint8).reshape(n, 32)[:, 20].long()
        model_turn = active & (to_play == model_player)
        valid = eng.valid_moves(roots)
        legal = valid.sum(1).cpu().tolist()
        budgets = torch.tensor([_n_searches(int(k), num_read) for k in legal], dtype=torch.int32, device=dev)
        budget = int(budgets[active].max())
        reads = torch.where(model_turn, budgets, torch.full((n,), -1, dtype=torch.int32, device=dev))
        noise = None
        if alpha > 0:
            g_ = torch._standard_gamma(torch.full((n, eng.A), float(alpha), dtype=torch.float64, device=dev), generator=gen)
            noise = g_ / g_.sum(-1, keepdim=True) * valid
        eng.run_search(reads, evaluator, noise=noise, coeff=coeff, max_reads=budget)
        v = eng.root_visits().double()
        probs = (v / v.max(1, keepdim=True).values.clamp_min(1.0)) ** (1.0 / temperature)
        probs = torch.where(model_turn.unsqueeze(1), probs, valid.double())
        probs = probs + (probs.sum(1, keepdim=True) == 0).double()
        m_model = torch.multinomial(probs, 1, generator=gen).reshape(-1)
        mm, mg = solver.moves(roots)
        best = ((mm != ILLEGAL) & (mm == mg.unsqueeze(1))).double()
        best = best + (best.sum(1, keepdim=True) == 0).double()
        m_solver = torch.multinomial(best, 1, generator=gen).reshape(-1)
        moves = torch.where(active, torch.where(model_turn, m_model, m_solver), torch.full_like(m_model, -1)).int()
        played = mm.gather(1, moves.clamp_min(0).long().unsqueeze(1)).squeeze(1)
        blunders += (model_turn & (torch.sign(played) < torch.sign(mg))).sum()
        model_moves += model_turn.sum()
        hist_states.append(roots[:n_games])
        hist_moves.append(moves[:n_games])
        hist_model.append(model_turn[:n_games])
        eng.advance_roots(moves, reuse=bool(sp.reuse_mcts_tree))
    final = eng.root_states()
    res = eng.result(final)
    eng.status()
    winner = final.view(torch.uint8).reshape(n, 32)[:, 21].long()  # just_played of the terminal state
    result = torch.where(res == 0, 0, torch.where(winner == model_player, 1, -1)).to(torch.int8)[:n_games]
    return {"wins": int((result == 1).sum()), "draws": int((result == 0).sum()), "losses": int((result == -1).sum()),
            "model_moves": int(model_moves), "blunders": int(blunders), "result": result,
            "states": torch.stack(hist_states), "moves": torch.stack(hist_moves), "model": torch.stack(hist_model)}
