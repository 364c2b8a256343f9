"""Self-play drivers (reference: self_play.py).

SelfPlay         drop-in for self_play.py:19-156: one game at a time through the mcts drop-in and any
                 `async nn(game_state)`; same temperature / np.random.choice protocol, same played_games
                 layout and the same get_datasets() DataFrame.
BatchedSelfPlay  the B200 path: `n_games` games in lock-step on one Engine, leaf evaluation by a
                 device-resident evaluator, per-game legacy RNG streams on the host so that a game
                 played with seed s is move-for-move the game the reference plays after
                 np.random.seed(s).
generate_games   self_play.py:291-306 re-targeted: games are sharded by index over the ranks of
                 torch.distributed (one process per GPU) instead of an mp.Pool; the sample rows are
                 gathered to rank 0 (the reference appends to an HDF file under a lock).
"""
import logging
import math
import time

import ctypes as C

import numpy as np
import pandas as pd
import torch

from . import mcts
from ._capi import RESULT_NONE, STATE_DTYPE
from .dots_boxes.dots_boxes_game import BoxesState

logger = logging.getLogger(__name__)


def _apply_temperature(visit_counts, temperature):
    # self_play.py:32-33 (float64)
    probs = (visit_counts / visit_counts.max()) ** (1 / temperature)
    return probs / probs.sum()


def _n_searches(n_valid, num_read):
    return min(4 * math.factorial(n_valid), num_read)  # self_play.py:64-65


def _game_outcomes(final, result, margin):
    """Per game (int8 tensors [n]): the player whose sample rows get z = +outcome, and the outcome; every other row of
    the game gets -outcome.  A game played out: just_played of its terminal state and its result.  A game adjudicated
    at a root, or played out exactly from it by the asynchronous loop, whose tree keeps that root (margin != ILLEGAL,
    the root's final margin): that root's player to move and sign(margin)."""
    from .solver import ILLEGAL
    raw = final.view(torch.uint8).reshape(-1, 32)
    adj = margin != ILLEGAL
    player = torch.where(adj, raw[:, 20], raw[:, 21]).to(torch.int8)
    outcome = torch.where(adj, torch.sign(margin), result.to(torch.int8))
    return player, outcome


def _hist_outcomes(h):
    """_game_outcomes of a device-resident history: adjudicated games (h["margin"]) and games played out exactly by the
    asynchronous loop (h["exact_margin"]; the two modes exclude each other)."""
    margin = h["margin"]
    if h.get("exact_margin") is not None:
        margin = torch.where(h["exact_margin"] != -128, h["exact_margin"], margin)
    return _game_outcomes(h["final"], h["result"], margin)


def _dataset(rows, generation, with_features):
    """The DataFrame of self_play.py:95-156 from row dicts (same columns, dtypes and MultiIndex)."""
    n = len(rows)
    players = np.asarray([r["player"] for r in rows], dtype=np.int8)
    if isinstance(generation, (list, tuple)):
        gen = np.zeros(n, dtype=np.int16)
        gen[players == 0] = generation[0]
        gen[players == 1] = generation[1]
    else:
        gen = np.asarray([generation] * n, dtype=np.int16)
    cols = {"generation": gen, "game_idx": np.asarray([r["game_idx"] for r in rows], dtype=np.int16),
            "move_idx": np.asarray([r["move_idx"] for r in rows], dtype=np.int16),
            "move": np.asarray([-1 if r["move"] is None else r["move"] for r in rows]).astype(np.int16),
            "player": players}
    df = pd.DataFrame(cols)
    if with_features:
        feats = np.stack([r["features"] for r in rows], axis=0) if n else np.zeros((0, 0), np.int16)
        df = df.join(pd.DataFrame(feats, columns=["x_" + str(i) for i in range(feats.shape[1])], index=df.index))
    pol = np.stack([r["pi"] for r in rows], axis=0) if n else np.zeros((0, 0))
    df = df.join(pd.DataFrame(pol, columns=["pi_" + str(i) for i in range(pol.shape[1])], index=df.index))
    df = df.join(pd.DataFrame(np.asarray([r["z"] for r in rows])[:, np.newaxis], columns=["z"], index=df.index))
    stats = pd.DataFrame.from_records([r["stats"] for r in rows], columns=["max_deepness", "tree_size", "terminal_count", "q_value"],
                                      index=df.index)
    df = df.join(stats.astype({"max_deepness": np.int16, "tree_size": np.int32, "terminal_count": np.int32, "q_value": np.float32}))
    df.set_index(["generation", "game_idx", "move_idx"], inplace=True)
    return df


class SelfPlay:
    """self_play.py:19-156"""

    def __init__(self, nn, params):
        self.played_games = []
        self.params = params
        self.nn = nn
        self.player_change_callback = lambda player: None

    async def get_next_move(self, root_node, nb_mcts_searches, temperature, dirichlet):
        mp = self.params.self_play.mcts
        visit_counts = await mcts.UCT_search(root_node, nb_mcts_searches, self.nn, mp.mcts_cpuct, mp.max_async_searches, dirichlet)
        probs = _apply_temperature(visit_counts, temperature)
        return np.random.choice(probs.shape[0], 1, p=probs)[0]

    async def play_game(self, game_state, idx):
        temperature = None
        seq = []
        root = mcts.create_root_uct_node(game_state)
        i = -1
        while not root.is_terminal:
            i += 1
            self.player_change_callback(root.game_state.to_play)
            params = self.params
            if i in params.self_play.mcts.temperature:
                temperature = params.self_play.mcts.temperature[i]
            n_valid = len(root.game_state.get_valid_moves(as_indices=True))
            move = await self.get_next_move(root, _n_searches(n_valid, params.self_play.mcts.mcts_num_read), temperature,
                                            params.self_play.noise)
            seq.append(root)
            root = mcts.init_mcts_tree(root, move, reuse_tree=params.self_play.reuse_mcts_tree)
        seq.append(root)
        self.played_games.append((idx, seq, root.game_state.get_result()))

    async def play_games(self, game_state, games_idxs, show_progress=False):
        for idx in games_idxs:
            if show_progress:
                print(".", end="", flush=True)
            await self.play_game(game_state, idx)

    def get_games_moves(self):
        moves, visit_counts = [], []
        for _, seq, _ in self.played_games:
            for node in seq[1:]:
                moves.append(node.move)
                visit_counts.append(node.child_number_visits)
        return moves, np.asarray(visit_counts, dtype=float)

    def set_player_change_callback(self, cb):
        self.player_change_callback = cb

    def get_datasets(self, generation, with_features=True):
        rows = []
        for game_idx, seq, z in self.played_games:
            winner = seq[-1].game_state.just_played
            for move_i, node in enumerate(seq[:-1]):
                vis = node.child_number_visits
                vs = vis.sum()
                rows.append({"game_idx": game_idx, "move_idx": move_i, "move": node.move, "player": node.game_state.to_play,
                             "z": z if node.game_state.to_play == winner else -z, "stats": tuple(node.get_tree_stats()),
                             "pi": vis / (vs or 1.0),
                             "features": node.game_state.get_features().ravel() if with_features else None})
        return _dataset(rows, generation, with_features)


class BatchedSelfPlay:
    """`engine.n_games` self-play games in lock-step on one GPU.

    evaluator(engine): fills engine.priors / engine.values from engine.planes (dotsboxesaz_b200.nn.DeviceEvaluator
    or engine.FakeNetEvaluator).  seeds: one legacy-MT19937 seed per game; per move the stream yields the
    Dirichlet draw (if alpha > 0) and then the uniform of np.random.choice, the reference's order (SURVEY 8c).

    adjudicate (default: params.self_play.adjudicate; None = off): max_free in 0 .. 16.  A game ends at the first root
    that is still going on and has at most max_free free edges; that root is not searched and gives no sample, and every
    row of the game takes its z from perfect play out of it (endgame.EndgameSolver): +outcome for the rows of the root's
    player to move, -outcome for the others.  So positions with f <= max_free leave the training data.  The natural
    evaluator to pair it with is EndgameEvaluator(inner, EndgameSolver(engine, m)) with m >= max_free, so that the net
    is never asked about the positions it no longer trains on (not enforced).  Games that end at a majority earlier are
    played as without adjudication.

    exact_endgame (default: params.self_play.exact_endgame; None = off): max_free in 0 .. 16, the alternative to
    adjudicate that keeps those positions (DESIGN.md §14).  From the first root that is still going on and has at most
    max_free free edges, the game is played out without a search: every root gives a sample row whose visits are 1 on the
    optimal moves and 0 elsewhere (so pi is uniform over them; exact_policy "outcome" or "margin" picks outcome- or
    margin-optimal moves), with zero tree statistics and q, and the move is drawn from that row by the path's usual
    draw law (temperature has no effect, no Dirichlet noise is drawn).  Every row's z is the played-out result, which
    optimal play keeps equal to the root's exact outcome.  Up to that root a game is the same game as without the
    mode.  adjudicate and exact_endgame exclude each other.
    """

    def __init__(self, engine, evaluator, params, graph_waves=16, pending=None, adaptive=None, adjudicate=None, exact_endgame=None,
                 exact_policy="outcome"):
        self.eng = engine
        self.ev = evaluator
        self.params = params
        self.graph_waves = graph_waves
        # adaptive wave loop (Engine.run_search): on by default when the engine has an eval cache, where the number of
        # waves a search needs is not known in advance
        self.adaptive = bool(engine.eval_cache_log2) if adaptive is None else bool(adaptive)
        # simulations in flight per tree: the reference's max_async_searches, capped by what the engine was built for
        want = params.self_play.mcts.max_async_searches if pending is None else pending
        self.pending = max(1, min(int(want or 1), engine.max_pending))
        self.played_games = []
        self.rows = []
        self.total_sims = 0
        m = params.self_play.get("adjudicate", None) if adjudicate is None else adjudicate
        self.endgame = None
        if m is not None:
            from .endgame import EndgameSolver
            if not 0 <= int(m) <= 16:
                raise ValueError("adjudicate must be a max_free in 0 .. 16 or None, got %r" % (m,))
            self.endgame = EndgameSolver(engine, int(m))
        x = params.self_play.get("exact_endgame", None) if exact_endgame is None else exact_endgame
        self.exact = None
        self.exact_policy = exact_policy
        if x is not None:
            from .endgame import EndgameSolver
            if not 0 <= int(x) <= 16:
                raise ValueError("exact_endgame must be a max_free in 0 .. 16 or None, got %r" % (x,))
            if self.endgame is not None:
                raise ValueError("adjudicate and exact_endgame exclude each other: set one of them")
            if exact_policy not in ("outcome", "margin"):
                raise ValueError("exact_policy must be 'outcome' or 'margin', got %r" % (exact_policy,))
            self.exact = EndgameSolver(engine, int(x))

    def play_games(self, games_idxs, seeds=None, start_states=None, with_features=True):
        eng, sp = self.eng, self.params.self_play
        n = eng.n_games
        games_idxs = list(games_idxs)
        assert len(games_idxs) <= n, "more games than engine slots"
        active = np.zeros(n, dtype=bool)
        active[:len(games_idxs)] = True
        seeds = list(seeds) if seeds is not None else list(games_idxs)
        rngs = [np.random.RandomState(s) for s in seeds] + [None] * (n - len(seeds))
        alpha, coeff = sp.noise
        num_read = sp.mcts.mcts_num_read
        temp_sched = sp.mcts.temperature
        eng.set_cpuct(sp.mcts.mcts_cpuct)
        eng.reset_roots(start_states)
        A = eng.A
        temperature = [None] * n
        hist = [[] for _ in range(n)]  # per game: row dicts of every searched root
        moves_played = [[] for _ in range(n)]
        margin = np.full(n, -128, dtype=np.int8)  # final margin of the root a game was adjudicated at, -128 (ILLEGAL) if none
        exact_seen = np.zeros(n, dtype=bool)      # games that reached exact play
        exact_rows = 0
        move_i = -1
        while active.any():
            move_i += 1
            roots = eng.root_states()
            valid = eng.valid_moves(roots).cpu().numpy()
            res = eng.result(roots).cpu().numpy()
            feats = eng.features(roots, torch.int16).cpu().numpy().reshape(n, -1) if with_features else None
            roots_np = eng.states_to_numpy(roots)
            active &= (res == RESULT_NONE)
            if self.endgame is not None:
                due = active & (self.endgame.free_edges(roots).cpu().numpy() <= self.endgame.max_free)
                if due.any():
                    idx = np.flatnonzero(due)
                    margin[idx] = self.endgame.margin(roots[torch.from_numpy(idx).to(roots.device)].contiguous()).cpu().numpy()
                    active &= ~due
            if not active.any():
                break
            due = np.zeros(n, dtype=bool)  # games in exact play: no search, visits = their optimal moves
            if self.exact is not None:
                due = active & (self.exact.free_edges(roots).cpu().numpy() <= self.exact.max_free)
                if due.any():
                    idx = np.flatnonzero(due)
                    opt = np.zeros((n, A), dtype=np.int32)
                    opt[idx] = self.exact.optimal_moves(roots[torch.from_numpy(idx).to(roots.device)].contiguous(),
                                                        self.exact_policy).cpu().numpy()
                    exact_seen |= due
                    exact_rows += int(due.sum())
            reads = np.full(n, -1, dtype=np.int32)
            noise = np.zeros((n, A), dtype=np.float64) if alpha > 0 else None
            for g in np.flatnonzero(active):
                if move_i in temp_sched:
                    temperature[g] = temp_sched[move_i]
                if due[g]:
                    continue
                reads[g] = _n_searches(int(valid[g].sum()), num_read)
                if alpha > 0:
                    noise[g] = rngs[g].dirichlet(np.ones(A) * alpha, 1).ravel() * valid[g]
            if (reads >= 0).any():
                eng.run_search(torch.from_numpy(reads), self.ev, noise=None if noise is None else torch.from_numpy(noise),
                               coeff=coeff, max_reads=int(reads.max()), graph_waves=self.graph_waves, pending=self.pending,
                               adaptive=self.adaptive)
            vis = eng.root_visits().cpu().numpy()
            stats, _rW, q = (x.cpu().numpy() for x in eng.tree_stats())
            if due.any():
                vis[due] = opt[due]
                stats[due] = 0
                q[due] = 0.0
            moves = np.full(n, -1, dtype=np.int32)
            for g in np.flatnonzero(active):
                probs = vis[g] / vis[g].sum() if due[g] else _apply_temperature(vis[g], temperature[g])
                r = rngs[g]
                moves[g] = r.choice(A, 1, p=probs)[0]
                hist[g].append({"game_idx": games_idxs[g], "move_idx": move_i, "move": moves_played[g][-1] if moves_played[g] else None,
                                "player": int(roots_np["to_play"][g]), "visits": vis[g].copy(),
                                "stats": (int(stats[g][1]), int(stats[g][2]), int(stats[g][3]), np.float32(q[g])),
                                "features": feats[g].copy() if with_features else None})
                moves_played[g].append(int(moves[g]))
                self.total_sims += int(stats[g][0]) if False else 0
            eng.advance_roots(moves, reuse=bool(sp.reuse_mcts_tree))
        info = eng.status()
        self.total_sims = info["sims"]
        info["adjudicated"] = int((margin[:len(games_idxs)] != -128).sum())
        info["exact_games"] = int(exact_seen[:len(games_idxs)].sum())
        info["exact_rows"] = exact_rows
        final = eng.root_states()
        winners, outcomes = (x.cpu().numpy() for x in _game_outcomes(final, eng.result(final), torch.from_numpy(margin).to(final.device)))
        for g in range(len(games_idxs)):
            z = int(outcomes[g])
            winner = int(winners[g])
            for r in hist[g]:
                vs = r["visits"].sum()
                r["pi"] = r["visits"] / (vs or 1.0)
                r["z"] = z if r["player"] == winner else -z
            self.rows.extend(hist[g])
            self.played_games.append((games_idxs[g], moves_played[g], [r["visits"] for r in hist[g]], z))
        return self.played_games

    def play_games_device(self, games_idxs, seed=0, start_states=None, with_features=True):
        """Throughput mode: the whole game loop stays on the device -- Dirichlet noise pre-drawn for every move
        (the reference draws it over ALL A entries and only then multiplies by the legal mask, mcts.py:220-223, so it
        does not depend on the position), temperature sampling with torch.multinomial, re-rooting with the sampled
        moves, samples accumulated in HBM -- and nothing synchronises with the host between moves.  Same algorithm
        and hyper-parameters as play_games(); the random streams differ (one device generator instead of one legacy
        NumPy stream per game), so games are not seed-identical to the reference's."""
        eng, sp = self.eng, self.params.self_play
        n, A, dev = eng.n_games, eng.A, eng.device
        games_idxs = list(games_idxs)
        assert len(games_idxs) == n, "play_games_device fills every engine slot"
        alpha, coeff = sp.noise
        num_read = sp.mcts.mcts_num_read
        temp_sched = sp.mcts.temperature
        n_edges = eng.L * (eng.C + 1) + eng.C * (eng.L + 1)
        eng.set_cpuct(sp.mcts.mcts_cpuct)
        eng.reset_roots(start_states)
        gen = torch.Generator(device=dev)
        gen.manual_seed(int(seed))
        roots0 = eng.root_states()
        played0 = int((~eng.valid_moves(roots0[:1])).sum().item()) - (A - n_edges)  # plies already on the board
        n_moves = n_edges - played0
        noise_all = None
        if alpha > 0:
            g = torch._standard_gamma(torch.full((n_moves, n, A), float(alpha), dtype=torch.float64, device=dev), generator=gen)
            noise_all = g / g.sum(-1, keepdim=True)
        temperature = None
        hist_states, hist_visits, hist_active, hist_moves, hist_stats, hist_q = [], [], [], [], [], []
        margin = torch.full((n,), -128, dtype=torch.int8, device=dev)  # final margin of an adjudicated game's root, else ILLEGAL
        solver = self.endgame if self.endgame is not None else self.exact
        full = solver.full_states(n) if solver is not None else None
        exact_seen = torch.zeros((n,), dtype=torch.bool, device=dev)     # games that reached exact play
        exact_rows = torch.zeros((), dtype=torch.int64, device=dev)
        for move_i in range(n_moves):
            if move_i in temp_sched:
                temperature = float(temp_sched[move_i])
            roots = eng.root_states()
            valid = eng.valid_moves(roots)
            active = eng.result(roots) == RESULT_NONE
            if self.endgame is not None:
                # roots reaching f <= max_free now: solved once (the other rows solve the f = 0 full board) and out of play
                active &= margin == -128
                due = active & (self.endgame.free_edges(roots) <= self.endgame.max_free)
                margin = torch.where(due, self.endgame.margin(torch.where(due.unsqueeze(1), roots, full).contiguous()), margin)
                active &= ~due
            exact = None
            if self.exact is not None:
                # roots in exact play: not searched, their visit row is their optimal moves (the other rows solve the full board)
                exact = active & (self.exact.free_edges(roots) <= self.exact.max_free)
                opt = self.exact.optimal_moves(torch.where(exact.unsqueeze(1), roots, full).contiguous(), self.exact_policy)
                exact_seen |= exact
                exact_rows += exact.sum()
            k = n_moves - move_i  # legal moves left: one edge is played per move
            searched = active if exact is None else active & ~exact
            reads = torch.where(searched, torch.full((n,), _n_searches(k, num_read), dtype=torch.int32, device=dev),
                                torch.full((n,), -1, dtype=torch.int32, device=dev))
            noise = noise_all[move_i] * valid if noise_all is not None else None
            eng.run_search(reads, self.ev, noise=noise, coeff=coeff, max_reads=_n_searches(k, num_read), graph_waves=self.graph_waves,
                           pending=self.pending, adaptive=self.adaptive)
            vis = eng.root_visits()
            stats, _rw, q = eng.tree_stats()
            if exact is not None:
                vis = torch.where(exact.unsqueeze(1), opt.int(), vis)
                stats = torch.where(exact.unsqueeze(1), torch.zeros_like(stats), stats)
                q = torch.where(exact, torch.zeros_like(q), q)
            v = vis.double()
            probs = (v / v.max(1, keepdim=True).values.clamp_min(1.0)) ** (1.0 / temperature)
            probs = torch.where(active.unsqueeze(1), probs, valid.double())  # finished games: any legal filler, ignored below
            probs = probs + (probs.sum(1, keepdim=True) == 0).double()       # ... or a dummy row if the board is full
            moves = torch.multinomial(probs, 1, generator=gen).reshape(-1).int()
            moves = torch.where(active, moves, torch.full_like(moves, -1))
            hist_states.append(roots); hist_visits.append(vis); hist_active.append(active); hist_moves.append(moves)
            hist_stats.append(stats); hist_q.append(q)
            eng.advance_roots(moves, reuse=bool(sp.reuse_mcts_tree))
        final = eng.root_states()
        res = eng.result(final)
        info = eng.status()  # the only host synchronisation of the whole batch of games
        self.total_sims = info["sims"]
        info["adjudicated"] = int((margin != -128).sum())
        info["exact_games"] = int(exact_seen.sum())
        info["exact_rows"] = int(exact_rows)
        self._device_hist = dict(states=hist_states, visits=hist_visits, active=hist_active, moves=hist_moves, stats=hist_stats,
                                 q=hist_q, final=final, result=res, margin=margin, games_idxs=games_idxs, with_features=with_features,
                                 noise=noise_all)  # the pre-drawn Dirichlet samples [move, game, A]: a run can be replayed
        return info

    def play_games_async(self, games_idxs, seed=0, start_states=None, with_features=True):
        """play_games_device() without the per-move lock-step: every game runs at its own pace.  A tree whose search has
        finished samples its move, re-roots and starts its next search at the next check (once per CUDA-graph replay)
        while the other trees are still searching, so no game waits for the slowest search of each move -- the batch
        takes as long as its slowest GAME, not as the sum of the slowest searches.  Same algorithm, hyper-parameters,
        per-game move sequence semantics and sample layout as play_games_device(); the moves are drawn from the same kind
        of device generator but in a different order, so individual games differ between the two.

        Needs the adaptive wave loop's machinery (compact rows, batch ladder, one simulation in flight per tree)."""
        eng, sp = self.eng, self.params.self_play
        n, A, dev = eng.n_games, eng.A, eng.device
        games_idxs = list(games_idxs)
        assert len(games_idxs) == n, "play_games_async fills every engine slot"
        assert self.pending == 1 and self.graph_waves > 0, "play_games_async needs max_pending_evals == 1 and CUDA graphs"
        alpha, coeff = sp.noise
        num_read = sp.mcts.mcts_num_read
        temp_sched = sp.mcts.temperature
        n_edges = eng.L * (eng.C + 1) + eng.C * (eng.L + 1)
        eng.set_cpuct(sp.mcts.mcts_cpuct)
        eng.reset_roots(start_states)
        gen = torch.Generator(device=dev)
        gen.manual_seed(int(seed))
        roots0 = eng.root_states()
        played0 = int((~eng.valid_moves(roots0[:1])).sum().item()) - (A - n_edges)  # plies already on the board
        n_moves = n_edges - played0
        if alpha > 0:
            g = torch._standard_gamma(torch.full((n_moves, n, A), float(alpha), dtype=torch.float64, device=dev), generator=gen)
            noise_all = g / g.sum(-1, keepdim=True)
        else:
            noise_all = torch.zeros((n_moves, n, A), dtype=torch.float64, device=dev)
        # per move index: temperature (piecewise constant schedule); per number of legal moves: simulation budget
        temps, t_cur = [], None
        for m in range(n_moves):
            t_cur = float(temp_sched[m]) if m in temp_sched else t_cur
            temps.append(t_cur)
        inv_temp = 1.0 / torch.tensor(temps, dtype=torch.float64, device=dev)
        reads_by_k = torch.tensor([_n_searches(k, num_read) if k > 0 else 0 for k in range(n_edges + 1)], dtype=torch.int32, device=dev)
        h_states = torch.zeros((n_moves, n, 4), dtype=torch.int64, device=dev)
        h_visits = torch.zeros((n_moves, n, A), dtype=torch.int32, device=dev)
        h_active = torch.zeros((n_moves, n), dtype=torch.bool, device=dev)
        h_moves = torch.full((n_moves, n), -1, dtype=torch.int32, device=dev)
        h_stats = torch.zeros((n_moves, n, 8), dtype=torch.int32, device=dev)
        h_q = torch.zeros((n_moves, n), dtype=torch.float32, device=dev)
        move_idx = torch.zeros((n,), dtype=torch.int64, device=dev)
        searching = torch.ones((n,), dtype=torch.int8, device=dev)
        moves = torch.full((n,), -1, dtype=torch.int32, device=dev)
        left_dev = torch.zeros((1,), dtype=torch.int32, device=dev)
        margin = torch.full((n,), -128, dtype=torch.int8, device=dev)  # final margin of an adjudicated game's root, else ILLEGAL
        exact_margin = torch.full((n,), -128, dtype=torch.int8, device=dev)  # ... of the root a game was played out from, else ILLEGAL
        u_all = torch.rand((n_moves, n), dtype=torch.float64, device=dev, generator=gen)  # one uniform per (move, game): the draw of the move

        eng.pending = 1
        eng.set_mode(True, eng.max_inline)
        if eng._noise_buf is None:
            eng._noise_buf = torch.zeros((n, A), dtype=torch.float64, device=dev)
        noise_buf = eng._noise_buf
        noise_arg = noise_buf if alpha > 0 else None  # alpha <= 0: the reference mixes the scalar 0.0 in (float32 arithmetic)
        graphs = eng._ladder_graphs(self.ev, self.graph_waves, noise_arg, coeff, short_tail=False)  # a small batch is no tail here
        ladder = eng._ladder(self.ev)
        per_wave = 1 + int(getattr(self.ev, "engine_launches", 0))
        reads = eng._num_reads  # the array begin() hands to the engine: written in place by the restart kernel
        from ._capi import SelfplayBuffers
        ptr = lambda t: C.c_void_p(t.data_ptr())
        bufs = SelfplayBuffers(n_moves=n_moves, inv_temp=ptr(inv_temp), uniforms=ptr(u_all), noise=ptr(noise_all) if alpha > 0 else None,
                               reads_by_k=ptr(reads_by_k), searching=ptr(searching), move_idx=ptr(move_idx), moves=ptr(moves),
                               h_states=ptr(h_states), h_visits=ptr(h_visits), h_active=ptr(h_active), h_moves=ptr(h_moves),
                               h_stats=ptr(h_stats), h_q=ptr(h_q), noise_buf=ptr(noise_buf), reads=ptr(reads), left=ptr(left_dev))
        keep = (bufs, inv_temp, reads_by_k, u_all, noise_all)  # the kernels hold raw pointers: these tensors live until the loop ends
        adj, ex = self.endgame, self.exact

        eng.selfplay_restart(bufs, first=True)  # every tree begins its first search ...
        if adj is not None:
            adj.adjudicate(bufs, margin, first=True)  # ... unless its start state is adjudicated already
        if ex is not None:
            ex.play_out(bufs, exact_margin, self.exact_policy, first=True)  # ... or is played out exactly already
        eng.begin(reads, noise_arg, coeff, 1)

        def finish():
            """Trees whose search has finished: record the sample, draw the move (k_selfplay_pick), re-root
            (k_advance_roots), budget and noise of the next search (k_selfplay_restart), end the games whose new root is
            adjudicated (k_selfplay_adjudicate, with adjudication on) or play them out exactly (k_selfplay_exact_endgame,
            with exact_endgame on), begin the other searches (k_search_begin).  Four or five launches on in-place state,
            captured as one CUDA graph."""
            eng.selfplay_pick(bufs)
            eng.advance_roots(moves, reuse=bool(sp.reuse_mcts_tree))
            eng.selfplay_restart(bufs)
            if adj is not None:
                adj.adjudicate(bufs, margin)
            if ex is not None:
                ex.play_out(bufs, exact_margin, self.exact_policy)
            eng.begin(reads, noise_arg, coeff, 1)

        # capture_begin / capture_end directly: the torch.cuda.graph() context empties the caching allocator (and the pinned
        # host cache) on entry, after which this call's next allocations -- hundreds of MB of history and samples beside a
        # 70 GB node arena -- go back to the driver; that cost up to a second of a three-second batch, at random
        fgraph = torch.cuda.CUDAGraph()
        l0 = eng.n_launches
        main = torch.cuda.current_stream(dev)
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(main)
        with torch.cuda.stream(side):
            fgraph.capture_begin()
            try:
                finish()
            finally:
                fgraph.capture_end()
        main.wait_stream(side)
        finish_launches = eng.n_launches - l0  # engine kernels inside the finish graph
        eng.n_launches = l0
        stream = torch.cuda.current_stream(dev)
        counts = torch.zeros((64, 4), dtype=torch.int32).pin_memory()
        left = torch.zeros((64,), dtype=torch.int32).pin_memory()
        events = []
        rows, i = ladder[0], 0
        while True:
            graphs[rows].replay()
            eng._count_replay(graphs[rows])
            eng.n_launches += finish_launches
            slot = counts[i % 64]
            eng.lib.dbaz_search_wave_counts(eng._h, C.c_void_p(slot.data_ptr()), eng._stream())
            fgraph.replay()
            left[i % 64:i % 64 + 1].copy_(left_dev, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(stream)
            events.append((ev, slot, left[i % 64]))
            i += 1
            if len(events) >= 2:
                ev0, slot0, left0 = events.pop(0)
                ev0.synchronize()
                if int(left0) == 0:
                    break
                want = min(n, int(int(slot0[2]) * eng.ROW_MARGIN) + 32)
                rows = eng._pick_rows(ladder, want, id(self.ev))
        del fgraph
        final = eng.root_states()
        res = eng.result(final)
        info = eng.status()
        self.total_sims = info["sims"]
        info["adjudicated"] = int((margin != -128).sum())
        info["exact_games"] = int((exact_margin != -128).sum())
        info["exact_rows"] = 0
        if ex is not None:  # rows of positions with f <= max_free: every one of them was played out exactly
            rows = h_states.reshape(-1, 4)[h_active.reshape(-1)].contiguous()
            info["exact_rows"] = int((eng.valid_moves(rows).sum(1) <= ex.max_free).sum()) if rows.shape[0] else 0
        info["checks"] = i  # finish-graph replays of the batch
        self._device_hist = dict(states=list(h_states.unbind(0)), visits=list(h_visits.unbind(0)), active=list(h_active.unbind(0)),
                                 moves=list(h_moves.unbind(0)), stats=list(h_stats.unbind(0)), q=list(h_q.unbind(0)), final=final,
                                 result=res, margin=margin, exact_margin=exact_margin, games_idxs=games_idxs, with_features=with_features,
                                 noise=noise_all if alpha > 0 else None,  # pre-drawn Dirichlet samples [move, game, A]
                                 uniforms=u_all, inv_temp=inv_temp)              # ... and what drew the moves
        del keep
        return info

    def device_samples(self):
        """(planes int16 [R, 3, L+1, C+1], pi float64 [R, A], z float32 [R], game slot [R], move index [R]) of the last
        play_games_device() / play_games_async() call, still on the device, move by move and slot by slot within a move
        (positions that were not searched -- finished games -- are dropped).  One features call and one compaction for the
        whole history."""
        h, eng = self._device_hist, self.eng
        n = eng.n_games
        act = torch.stack(h["active"])                                   # [M, n]
        M = act.shape[0]
        states = torch.stack(h["states"]).reshape(M * n, 4)
        idx = torch.nonzero(act.reshape(-1)).reshape(-1)                 # row-major: move index, then slot
        sel = states[idx].contiguous()
        planes = eng.features(sel, torch.int16)
        v = torch.stack(h["visits"]).reshape(M * n, eng.A)[idx].double()
        pi = v / v.sum(1, keepdim=True).clamp_min(1.0)
        slot, mi = idx % n, idx // n
        to_play = sel.view(torch.uint8).reshape(-1, 32)[:, 20].to(torch.int8)
        winner, outcome = _hist_outcomes(h)
        z_final = outcome.float()[slot]
        z = torch.where(to_play == winner[slot], z_final, -z_final)
        return planes, pi, z, slot, mi

    def get_games_moves(self):
        if not self.played_games and getattr(self, "_device_hist", None) is not None:
            self._rows_from_device(False)
        moves, vcs = [], []
        for _, mv, vis, _ in self.played_games:
            moves.extend(mv)
            vcs.extend(vis)
        return moves, np.asarray(vcs, dtype=float)

    def get_datasets(self, generation, with_features=True):
        if not self.rows and getattr(self, "_device_hist", None) is not None:
            return self._dataset_from_device(generation, with_features)
        return _dataset(self.rows, generation, with_features)

    def _dataset_from_device(self, generation, with_features=True):
        """The DataFrame of self_play.py:95-156 straight from the device-resident history of play_games_device() /
        play_games_async(): the same columns, dtypes, MultiIndex and row order (game by game, move by move) as
        _dataset(_rows_from_device()), built from whole arrays instead of one Python dict per row."""
        h, eng = self._device_hist, self.eng
        n, A = eng.n_games, eng.A
        act = torch.stack(h["active"]).t().contiguous()                       # [n, M]
        sel = act.reshape(-1)
        M = act.shape[1]
        states = torch.stack(h["states"])                                     # [M, n, 4]
        to_play_mn = states.view(torch.uint8).reshape(M, n, 32)[:, :, 20]
        pick = lambda t: t.transpose(0, 1).reshape((n * M,) + tuple(t.shape[2:]))[sel].cpu().numpy()
        vis = pick(torch.stack(h["visits"]))
        stats = pick(torch.stack(h["stats"]))
        q = pick(torch.stack(h["q"]))
        player = pick(to_play_mn).astype(np.int8)
        mv = torch.stack(h["moves"])                                          # [M, n]: the move played FROM position m
        prev = torch.cat([torch.full_like(mv[:1], -1), mv[:-1]], 0)           # ... the one that LED to position m
        move = pick(prev).astype(np.int16)
        g_of = torch.arange(n, device=act.device).unsqueeze(1).expand(n, M).reshape(-1)[sel].cpu().numpy()
        m_of = torch.arange(M, device=act.device).unsqueeze(0).expand(n, M).reshape(-1)[sel].cpu().numpy()
        winner, res = (x.cpu().numpy() for x in _hist_outcomes(h))
        res = res.astype(np.int64)
        z = np.where(player == winner[g_of], res[g_of], -res[g_of])
        games = np.asarray(h["games_idxs"])
        if isinstance(generation, (list, tuple)):
            gen = np.where(player == 0, generation[0], generation[1]).astype(np.int16)
        else:
            gen = np.full(len(g_of), generation, dtype=np.int16)
        cols = {"generation": gen, "game_idx": games[g_of].astype(np.int16), "move_idx": m_of.astype(np.int16), "move": move, "player": player}
        if with_features:
            feats = torch.stack([eng.features(s, torch.int16) for s in h["states"]]).reshape(M, n, -1)
            feats = pick(feats)
            cols.update({"x_" + str(i): feats[:, i] for i in range(feats.shape[1])})
        vs = vis.sum(1, keepdims=True).astype(np.float64)
        pi = vis / np.where(vs == 0, 1.0, vs)
        cols.update({"pi_" + str(i): pi[:, i] for i in range(A)})
        cols["z"] = z
        cols["max_deepness"] = stats[:, 1].astype(np.int16)
        cols["tree_size"] = stats[:, 2].astype(np.int32)
        cols["terminal_count"] = stats[:, 3].astype(np.int32)
        cols["q_value"] = q.astype(np.float32)
        df = pd.DataFrame(cols)
        df.set_index(["generation", "game_idx", "move_idx"], inplace=True)
        return df

    def _rows_from_device(self, with_features=True):
        """Turn the device-resident history of play_games_device() into the row dicts of get_datasets()."""
        h, eng = self._device_hist, self.eng
        n = eng.n_games
        winner, res = (x.cpu().numpy() for x in _hist_outcomes(h))
        act = torch.stack(h["active"]).cpu().numpy()
        moves = torch.stack(h["moves"]).cpu().numpy()
        vis = torch.stack(h["visits"]).cpu().numpy()
        stats = torch.stack(h["stats"]).cpu().numpy()
        q = torch.stack(h["q"]).cpu().numpy()
        to_play = np.stack([eng.states_to_numpy(s)["to_play"] for s in h["states"]])
        feats = None
        if with_features:
            feats = torch.stack([eng.features(s, torch.int16) for s in h["states"]]).cpu().numpy().reshape(len(h["states"]), n, -1)
        for g in range(n):
            z = int(res[g])
            for m in range(act.shape[0]):
                if not act[m, g]:
                    continue
                v = vis[m, g]
                self.rows.append({"game_idx": h["games_idxs"][g], "move_idx": m, "move": int(moves[m - 1, g]) if m else None,
                                  "player": int(to_play[m, g]), "visits": v, "pi": v / (v.sum() or 1.0),
                                  "z": z if to_play[m, g] == winner[g] else -z,
                                  "stats": (int(stats[m, g][1]), int(stats[m, g][2]), int(stats[m, g][3]), np.float32(q[m, g])),
                                  "features": feats[m, g] if with_features else None})
            self.played_games.append((h["games_idxs"][g], [int(x) for x in moves[:, g] if x >= 0],
                                      [vis[m, g] for m in range(act.shape[0]) if act[m, g]], z))


class DualEvaluator:
    """Two nets, one per player, for the Elo arena (self_play.py:237-239 swaps the model on every move according to
    the player to move at the ROOT): both nets evaluate the wave and each game keeps the rows of the model that owns
    its current root.  `owner` (int8 [n_games], 0/1) is set by the driver before every search."""

    def __init__(self, ev0, ev1, engine):
        self.evs = (ev0, ev1)
        self.owner = torch.zeros((engine.n_games,), dtype=torch.bool, device=engine.device)
        self.engine_launches = getattr(ev0, "engine_launches", 0) + getattr(ev1, "engine_launches", 0)
        self._p0 = torch.empty_like(engine._priors)
        self._v0 = torch.empty_like(engine._values)

    def __call__(self, eng):
        rows = eng.n_rows
        self.evs[0](eng)
        self._p0[:rows].copy_(eng.priors)
        self._v0[:rows].copy_(eng.values)
        self.evs[1](eng)
        own1 = self.owner.repeat(eng.pending)  # row of slot k of tree t = k * n_games + t
        eng.priors.copy_(torch.where(own1.unsqueeze(1), eng.priors, self._p0[:rows]))
        eng.values.copy_(torch.where(own1, eng.values, self._v0[:rows]))


def compute_elo(elo_params, params, generations, elos, models=None, engine=None):
    """self_play.py:309-344: `elo_params.n_games` games between the nets of two generations (no tree reuse, no noise,
    more reads: elo_params.self_play_override), colours alternated between games, ratings updated with elo_rating2.
    models: the two nn.Modules (else built from params[i].nn.model_class and loaded from their checkpoints).
    Returns (elo0, elo1, share of games won by generations[1])."""
    import copy
    from . import engine as _engine
    from .nn import make_evaluator
    from .utils.utils import elo_rating2
    params = [copy.deepcopy(p) for p in params]
    for p in params:
        p.self_play.merge(elo_params.self_play_override)
    n = int(elo_params.n_games)
    own_engine = engine is None
    if engine is None:
        engine = _engine.Engine(tuple(params[0].game.clazz.BOARD_DIM), n_games=n,
                                max_nodes=int(params[0].self_play.get("max_nodes_per_tree", 8192) or 8192))
    # The eval cache is keyed by the position alone: with two nets in play it would serve each player the other
    # generation's evaluations (the reference switches its LRU off for model comparison, self_play.py:230).  A caller's
    # engine gets its table back afterwards.  DualEvaluator also assumes row == slot * n_games + tree: no compact rows.
    saved_cache = engine.eval_cache_log2
    if saved_cache:
        engine.set_eval_cache(0)
    engine.set_mode(False, engine.max_inline)
    if models is None:
        models = []
        for p, g in zip(params, generations):
            m = p.nn.model_class(p)
            if g != 0:
                m.load_parameters(g, to_device=engine.device)
            models.append(m)
    dual = DualEvaluator(make_evaluator(models[0], engine), make_evaluator(models[1], engine), engine)
    sp = BatchedSelfPlay(engine, dual, params[0], pending=1)
    # player p of game g is generation (p + g) % 2: colours alternate between games (the reference shuffles by worker pid)
    swap = torch.arange(n, device=engine.device) % 2 == 1
    eng = engine
    eng.set_cpuct(params[0].self_play.mcts.mcts_cpuct)
    eng.reset_roots()
    alpha, coeff = params[0].self_play.noise
    temperature, move_i = None, -1
    gen = torch.Generator(device=eng.device)
    gen.manual_seed(int(elo_params.get("seed", 0) or 0))
    n_edges = eng.L * (eng.C + 1) + eng.C * (eng.L + 1)
    for move_i in range(n_edges):
        if move_i in params[0].self_play.mcts.temperature:
            temperature = float(params[0].self_play.mcts.temperature[move_i])
        roots = eng.root_states()
        active = eng.result(roots) == RESULT_NONE
        if not bool(active.any()):
            break
        to_play = roots.view(torch.uint8).reshape(n, 32)[:, 20].bool()
        dual.owner.copy_(to_play ^ swap)
        k = n_edges - move_i
        reads = torch.where(active, torch.full((n,), _n_searches(k, params[0].self_play.mcts.mcts_num_read), dtype=torch.int32,
                                               device=eng.device), torch.full((n,), -1, dtype=torch.int32, device=eng.device))
        noise = None
        if alpha > 0:
            g_ = torch._standard_gamma(torch.full((n, eng.A), float(alpha), dtype=torch.float64, device=eng.device), generator=gen)
            noise = g_ / g_.sum(-1, keepdim=True) * eng.valid_moves(roots)
        eng.run_search(reads, dual, noise=noise, coeff=coeff, max_reads=_n_searches(k, params[0].self_play.mcts.mcts_num_read))
        v = eng.root_visits().double()
        probs = (v / v.max(1, keepdim=True).values.clamp_min(1.0)) ** (1.0 / temperature)
        probs = torch.where(active.unsqueeze(1), probs, eng.valid_moves(roots).double())
        probs = probs + (probs.sum(1, keepdim=True) == 0).double()
        moves = torch.multinomial(probs, 1, generator=gen).reshape(-1).int()
        eng.advance_roots(torch.where(active, moves, torch.full_like(moves, -1)), reuse=bool(params[0].self_play.reuse_mcts_tree))
    final = eng.root_states()
    res = eng.result(final)
    eng.status()
    winner_player = final.view(torch.uint8).reshape(n, 32)[:, 21].bool()  # just_played of the terminal state
    decided = res != 0
    winner_gen = (winner_player ^ swap) & decided
    n1 = int(winner_gen.sum())
    n0 = int(decided.sum()) - n1
    elo0, elo1 = elo_rating2(elos[0], elos[1], n0, n1, K=30)
    print(f"generation {generations[0]}: wins={n0}, elo={elos[0]} -> {elo0}")
    print(f"generation {generations[1]}: wins={n1}, elo={elos[1]} -> {elo1}")
    if own_engine:
        engine.close()
    elif saved_cache:
        engine.set_eval_cache(saved_cache)
    return elo0, elo1, n1 / max(1, n0 + n1)


def shard_game_indices(n_games, rank, world):
    """Games are independent: rank r plays the indices i with i % world == r (self_play.py:184 does the
    same round-robin over devices with its worker pids)."""
    return list(range(rank, n_games, world))


def broadcast_model(model, src=0):
    """The reference hands new weights to its self-play workers through model_gen{g}.pt on disk
    (nn.py:272-273 -> self_play.py:188-190); here one flat NCCL/gloo broadcast of parameters + BN buffers."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return
    tensors = [p.data for p in model.parameters()] + [b.data for b in model.buffers()]
    by_dtype = {}
    for t in tensors:
        by_dtype.setdefault(t.dtype, []).append(t)
    for dt, ts in by_dtype.items():
        flat = torch.cat([t.reshape(-1) for t in ts])
        dist.broadcast(flat, src=src)
        off = 0
        for t in ts:
            t.copy_(flat[off:off + t.numel()].reshape(t.shape))
            off += t.numel()


def gather_samples(df, dst=0):
    """Replaces the locked HDF append (self_play.py:264-265): every rank's sample rows end up on rank `dst`."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return df
    out = [None] * dist.get_world_size() if dist.get_rank() == dst else None
    dist.gather_object(df, out, dst=dst)
    if dist.get_rank() != dst:
        return None
    return pd.concat(out).sort_index()


def eval_cache_log2_for(A, n_slots, max_nodes, device=None):
    """log2(entries) of the eval cache for an engine of `n_slots` trees that plays whole games: about 4096 slots per tree
    (a direct-mapped table wants a few slots per insert; measured on 3x3 with 32 768 games per GPU: 2^24 entries 38.7 M
    games/h, 2^25 41.0 M, 2^26 43.2 M, 2^27 45.2 M -- a game inserts ~900 positions, most of them shared with other games),
    within 40 % of the device's memory and what the node pools leave free.  Emptying the table costs nothing (a table
    epoch), so its size only costs memory."""
    cell = 16 * int(A)
    budget = 8 << 30
    try:
        total = torch.cuda.get_device_properties(device if device is not None else torch.cuda.current_device()).total_memory
        pools = int(n_slots) * int(max_nodes) * (32 + cell)
        budget = max(1 << 30, min(int(0.4 * total), total - pools - (24 << 30)))
    except Exception:  # no device to ask (CPU-only import): the conservative 8 GB
        pass
    want = max(1, 4096 * int(n_slots))
    return max(16, min(int(np.log2(budget / cell)), int(np.ceil(np.log2(want)))))


def default_eval_cache(params, n_slots=None, max_nodes=None, device=None):
    """log2(entries) of the engine's eval cache: `params.self_play.eval_cache_log2` if given (0 = none), else sized for
    the engine (eval_cache_log2_for) -- or, without an engine size, up to 8 GB worth (3x3: 2^24 entries of 512 bytes) --
    the role of the reference's `nn.max_cache_size` LRU (self_play.py:226-230).  (Only searches with one simulation in
    flight per tree use the table; generate_games builds its engine that way.)"""
    sp = params.self_play
    want = sp.get("eval_cache_log2", None)
    if want is not None:
        return int(want)
    L, C = tuple(params.game.clazz.BOARD_DIM)
    A = 2 * (L + 1) * (C + 1)
    if n_slots:
        return eval_cache_log2_for(A, n_slots, max_nodes or 8192, device)
    return max(16, int(np.log2((8 << 30) / (16 * A))))


def shard_engine(params, n_shard_games, device=None):
    """One engine per rank, sized for THIS rank's shard of a generation (never for the global game count) and meant to
    live for the whole coach run: its node pool and eval cache are raw device memory that only engine.close() returns."""
    from . import engine as _engine
    cap = int(params.self_play.get("concurrent_games", 4096) or 4096)
    n_chunks = max(1, -(-int(n_shard_games) // cap))
    slots = max(1, -(-int(n_shard_games) // n_chunks))  # equal chunks: the last one is short by less than n_chunks games
    max_nodes = int(params.self_play.get("max_nodes_per_tree", 8192) or 8192)
    return _engine.Engine(tuple(params.game.clazz.BOARD_DIM), n_games=slots, max_nodes=max_nodes,
                          eval_cache=default_eval_cache(params, slots, max_nodes, device), device=device)


def game_seed(base_seed, generation, game_idx):
    """Seed of one game's legacy-MT19937 stream: a function of (base seed, generation, game index), so that no two
    generations replay the same noise and move-sampling uniforms (the reference's workers never reseed either)."""
    return int(np.random.SeedSequence([int(base_seed), int(generation), int(game_idx)]).generate_state(1)[0])


def play_shard(params, generation, engine, evaluator, indices, want_frames=False):
    """This rank's games of one generation.  Returns (samples.SampleBatch on the engine's device, [DataFrame, ...] if
    want_frames, info dict).  Full-width batches run every game at its own pace (play_games_async: device RNG, samples stay
    in HBM); `params.self_play.rng == "host"` keeps one legacy NumPy stream per game (reference-exact games, host loop).
    A short last chunk is padded with throw-away games (index -1) so that it takes the same device-resident path."""
    from . import samples
    indices = list(indices)
    base_seed = int(params.self_play.get("seed", 0) or 0)
    host_rng = params.self_play.get("rng", "device") == "host"
    n = engine.n_games
    batches, frames = [], []
    info = {"sims": 0, "games": len(indices), "chunks": 0}
    for lo in range(0, len(indices), n):
        chunk = indices[lo:lo + n]
        sp = BatchedSelfPlay(engine, evaluator, params)
        if host_rng:
            sp.play_games(chunk, seeds=[game_seed(base_seed, generation, i) for i in chunk])
            df = sp.get_datasets(generation, True)
            batches.append(samples.batch_from_frame(df, engine.device, generation))
        else:
            padded = chunk + [-1] * (n - len(chunk))
            seed = game_seed(base_seed, generation, chunk[0])
            (sp.play_games_async if (sp.adaptive and sp.pending == 1 and sp.graph_waves > 0) else sp.play_games_device)(padded, seed=seed)
            batches.append(samples.batch_from_selfplay(sp, generation))
            df = None
            if want_frames:
                df = sp.get_datasets(generation, True)
                df = df[df.index.get_level_values("game_idx") >= 0]
        if want_frames:
            frames.append(df)
        info["sims"] += sp.total_sims
        info["chunks"] += 1
    return samples.SampleBatch.cat(batches), frames, info


def generate_games(hdf_file_name, generation, nn_class, n_games, params, n_workers=None, games_per_workers=10,
                   engine=None, evaluator=None, writer=None, return_batch=False):
    """self_play.py:291-306.  One process per GPU (torch.distributed), `n_games` sharded by index; every rank plays its
    shard on its own engine (play_shard), the (features, pi, z) rows are gathered to rank 0 as device tensors with one
    NCCL collective (samples.gather_batches -- the reference's locked HDF append, self_play.py:264-265), and the
    DataFrame of self_play.py:95-156 is only built for export: each rank hands its own rows to
    `writer(hdf_file_name, "fresh", df)` (default: a part of the replay store) unless
    `params.self_play.export_frames` is False.  Returns the DataFrame of this rank's rows (None without export), or
    with return_batch the tuple (df, gathered SampleBatch on rank 0 / None elsewhere, info)."""
    import torch.distributed as dist
    from . import samples
    from .nn import make_evaluator
    rank = dist.get_rank() if dist.is_available() and dist.is_initialized() else 0
    world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
    mine = shard_game_indices(n_games, rank, world)
    own_engine = engine is None
    if own_engine:
        engine = shard_engine(params, len(mine))
    try:
        engine.clear_eval_cache()  # cached evaluations belong to the previous generation's weights
        if evaluator is None:
            model = nn_class(params)
            if generation != 0:
                model.load_parameters(generation - 1, to_device=engine.device)
            broadcast_model(model.to(engine.device))
            evaluator = make_evaluator(model, engine)
        export = bool(params.self_play.get("export_frames", True))
        t0 = time.time()
        batch, frames, info = play_shard(params, generation, engine, evaluator, mine, want_frames=export)
        torch.cuda.synchronize(engine.device)
        info["play_s"] = time.time() - t0
        t0 = time.time()
        gathered = samples.gather_batches(batch, engine.F, engine.A, dst=0, device=engine.device)
        torch.cuda.synchronize(engine.device)
        info["gather_s"] = time.time() - t0
        df = None
        if export and frames:
            t0 = time.time()
            df = pd.concat(frames)
            df["training"] = np.zeros(len(df.index), dtype=np.int8)
            if writer is None:
                from .utils.utils import ReplayStore
                store = ReplayStore(hdf_file_name)
                writer = lambda f, k, d: store.append(k, d, part="r%03d" % rank)
            writer(hdf_file_name, "fresh", df)
            info["export_s"] = time.time() - t0
    finally:
        if own_engine:
            engine.close()
    return (df, gathered, info) if return_batch else df
