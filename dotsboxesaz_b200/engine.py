"""Host-side handle of the CUDA engine: batched game rules and lock-step tree search.

PyTorch is used for device memory, streams and CUDA graphs only; every rule and every tree
operation runs in the hand-written sm_100a kernels behind include/dbaz_b200.h.  There is no
CPU path: constructing an Engine without a CUDA device raises RuntimeError.
"""
import ctypes as C
import os

import numpy as np
import torch

from . import _capi
from ._capi import STATE_DTYPE, RESULT_NONE

_DTYPE_CODE = {torch.float32: _capi.F32, torch.float16: _capi.F16, torch.bfloat16: _capi.BF16, torch.int16: _capi.I16}


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


class EngineError(RuntimeError):
    pass


class TrunkConvPlan:
    """A trunk convolution bound to its buffers (Engine.nn_trunk_conv_plan): the host bytes the launch passes to the
    kernel, and the tensors they point to, kept alive with the plan."""

    def __init__(self, buf, tensors):
        self.buf = buf
        self.x, self.y, self.w, self.bias_pos, self.bias = tensors


def trunk_conv_taps(hi, wi, pad):
    """Tap table of the trunk convolution kernel (include/dbaz_b200.h: dbaz_nn_trunk_conv_taps); needs no device.
    Returns (ho, wo, taps, order): taps[p] = [(input position, 3 ky + kx), ...] in accumulation order, order = the output
    positions as the kernel hands them out."""
    out = (C.c_int32 * (2 + 11 * _capi.TRUNK_MAX_POS))()
    if _capi.load().dbaz_nn_trunk_conv_taps(int(hi), int(wi), int(pad), out) != 0:
        raise ValueError("trunk conv: unsupported grid %dx%d with padding %d" % (hi, wi, pad))
    v = list(out)
    ho, wo = v[0], v[1]
    taps = []
    for p in range(ho * wo):
        row = v[2 + 10 * p: 12 + 10 * p]
        taps.append([(e >> 8, e & 255) for e in row[1:1 + row[0]]])
    base = 2 + 10 * _capi.TRUNK_MAX_POS
    return ho, wo, taps, v[base: base + ho * wo]


class Engine:
    """One engine = one GPU's shard of concurrent games (`n_games` trees of at most `max_nodes` nodes).

    States are device tensors of shape [n, 4] int64 (32 packed bytes each, see STATE_DTYPE).
    """

    def __init__(self, board=(3, 3), n_games=1, max_nodes=8192, cpuct=(1.25, 19652), device=None, lut_size=0, max_pending=1,
                 eval_cache=0):
        if not torch.cuda.is_available():
            raise RuntimeError("dotsboxesaz_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.lib = _capi.load()
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("dotsboxesaz_b200 engines live on CUDA devices only")
        dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.device = torch.device("cuda", dev_index)
        cfg = _capi.Config(1, dev_index, int(board[0]), int(board[1]), int(n_games), int(max_nodes), int(lut_size), int(max_pending),
                           float(cpuct[0]), float(cpuct[1]))
        h = C.c_void_p()
        torch.cuda.init()
        if self.lib.dbaz_engine_create(C.byref(cfg), C.byref(h)) != 0:
            raise EngineError(self.lib.dbaz_last_error(None).decode())
        self._h = h
        info = (C.c_int32 * 8)()
        self.lib.dbaz_engine_info(self._h, info)
        self.L, self.C, self.A, self.F, self.n_games, self.max_nodes, self.node_bytes, self.max_pending = list(info)
        self.rows, self.cols = self.L + 1, self.C + 1
        self.cpuct = (float(cpuct[0]), float(cpuct[1]))
        # search I/O buffers (fixed addresses, so the wave loop can be captured in a CUDA graph).  One row per
        # in-flight simulation: row of slot k of tree t = k * n_games + t; a search with max_pending_evals = K uses
        # the first K * n_games rows (`self.n_rows`), evaluators work on the `[:n_rows]` views below.
        cap = n_games * self.max_pending
        self._priors = torch.zeros((cap, self.A), dtype=torch.float32, device=self.device)
        self._values = torch.zeros((cap,), dtype=torch.float32, device=self.device)
        self._leaf_states = torch.zeros((cap, 4), dtype=torch.int64, device=self.device)
        self._leaf_kind = torch.zeros((cap,), dtype=torch.int8, device=self.device)
        self.pending = 1
        self._batch_rows = None      # evaluator batch of the adaptive wave loop (None: pending * n_games)
        self._planes = None
        self._planes_base = None
        self._plane_cfg = None
        self._noise = None  # keeps the caller's noise buffer alive while the engine may read it
        self._num_reads = torch.zeros((n_games,), dtype=torch.int32, device=self.device)
        self._idle_reads = torch.full((n_games,), -1, dtype=torch.int32, device=self.device)
        self._noise_buf = None
        self._graphs = {}
        self._graph_cost = {}
        self._loops = {}             # one-graph-per-search loops (dbaz_search_loop_build) per ladder of captured graphs
        self._loop_pending = []      # (event, pinned replay counts, graphs of the ladder) of launches not yet folded in
        self._nl = 0                 # engine kernels enqueued (graph replays count the kernels they contain)
        self._nw = 0
        # Optional: the adaptive wave loop as ONE graph per search (WHILE / SWITCH conditional nodes, device-side rung
        # choice): no host wait inside a search.  DBAZ_LOOP=0 keeps the host-driven loop.
        self.device_loop = os.environ.get("DBAZ_LOOP", "1") != "0"
        self.set_planes(torch.float32, channels_last=False)
        self.n_sms = torch.cuda.get_device_properties(self.device).multi_processor_count
        # lock-step scheduling state (see set_mode / run_search(adaptive=True))
        self.compact = False
        self.max_inline = 0
        self.set_mode(False, 4)
        # captured wave loops bound the in-kernel chains by TIME (microseconds per tree and launch; 0 = by count only,
        # max_inline): see include/dbaz_b200.h, dbaz_search_set_chain_budget.  20 us measured best on configs[1] (8 .. 30 swept:
        # +3 % sims/s over the count of 4) and in self-play (+6 % games/h); results do not depend on it.
        self.chain_us = int(os.environ.get("DBAZ_CHAIN_US", "20"))
        self.eval_cache_log2 = 0
        self._counts_host = torch.zeros((64, 4), dtype=torch.int32).pin_memory()
        self._graph_pool = None
        self._eval_us = {}           # (id(evaluator), batch rows) -> measured microseconds per evaluator call
        self._loop_counts_host = None
        if eval_cache:
            self.set_eval_cache(eval_cache)

    # ------------------------------------------------------------ plumbing
    @property
    def n_launches(self):
        """Engine kernels enqueued so far (graph replays count the kernels they contain)."""
        self._fold_loop_counts()
        return self._nl

    @n_launches.setter
    def n_launches(self, v):
        self._fold_loop_counts()
        self._nl = int(v)

    @property
    def n_waves(self):
        """dbaz_search_step launches so far (graph replays count the waves they contain)."""
        self._fold_loop_counts()
        return self._nw

    @n_waves.setter
    def n_waves(self, v):
        self._fold_loop_counts()
        self._nw = int(v)

    def _fold_loop_counts(self):
        """Replays the device-driven loops ran since the last look: their per-rung counts arrive by an asynchronous copy."""
        while self._loop_pending:
            ev, counts, ladder, graphs = self._loop_pending.pop(0)
            ev.synchronize()
            for r, c in zip(ladder, counts.tolist()):
                launches, waves = self._graph_cost.get(id(graphs[r]), (0, 0))
                self._nl += int(c) * launches
                self._nw += int(c) * waves

    def _drop_loops(self):
        for loop, _, _ in self._loops.values():
            self.lib.dbaz_search_loop_destroy(self._h, C.c_uint64(loop))
        self._loops = {}

    def close(self):
        if getattr(self, "_h", None):
            try:
                torch.cuda.synchronize(self.device)
                self._drop_loops()
            except Exception:
                pass
            self.lib.dbaz_engine_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return C.c_uint64(torch.cuda.current_stream(self.device).cuda_stream)

    def _ck(self, rc, launches=1):
        self._nl += launches
        if rc != 0:
            raise EngineError(self.lib.dbaz_last_error(self._h).decode())

    def _states_arg(self, states):
        if states.dtype != torch.int64 or states.dim() != 2 or states.shape[1] != 4 or not states.is_contiguous() \
                or states.device != self.device:
            raise ValueError("states must be a contiguous int64 [n, 4] tensor on %s" % self.device)
        return states

    def set_cpuct(self, cpuct):
        """mcts.py:205 -- UCT_search re-assigns the PUCT constants on every call."""
        cpuct = (float(cpuct[0]), float(cpuct[1]))
        if cpuct != self.cpuct:
            self._ck(self.lib.dbaz_engine_set_cpuct(self._h, cpuct[0], cpuct[1]))
            self.cpuct = cpuct

    @property
    def n_rows(self):
        """Leaf rows the evaluator works on: max_pending_evals * n_games, or the (smaller) batch the adaptive wave
        loop of run_search() currently runs at."""
        return self.pending * self.n_games if self._batch_rows is None else self._batch_rows

    # ------------------------------------------- eval cache / scheduling mode
    def set_eval_cache(self, log2_entries):
        """Device table of 2**log2_entries cached evaluations keyed by get_hash() -- the engine's form of
        AsyncBatchedProxy's LRU (utils/proxies.py:23-26,35-43); 0 frees it.  Synchronises."""
        self._ck(self.lib.dbaz_cache_configure(self._h, int(log2_entries)), launches=0)
        self.eval_cache_log2 = int(log2_entries)
        self._drop_loops()
        self._graphs = {}  # captured step kernels carry the table pointer
        self._graph_pool = None  # the pool dies with its last graph

    def clear_eval_cache(self):
        """Forget all cached evaluations (after a weight update)."""
        self._ck(self.lib.dbaz_cache_clear(self._h, self._stream()), launches=0)

    def set_mode(self, compact=False, max_inline=0):
        """compact: leaves go to consecutive batch rows (see include/dbaz_b200.h); max_inline: bound on the
        simulations per tree and wave that finish without the evaluator (0 = unbounded)."""
        if (bool(compact), int(max_inline)) != (self.compact, self.max_inline):
            self._ck(self.lib.dbaz_search_set_mode(self._h, 1 if compact else 0, int(max_inline)), launches=0)
            self.compact, self.max_inline = bool(compact), int(max_inline)

    def set_chain_budget(self, microseconds):
        """Time bound of the in-kernel chains for the launches that follow (0 = off): include/dbaz_b200.h,
        dbaz_search_set_chain_budget.  The captured wave loops set their own (self.chain_us)."""
        self._ck(self.lib.dbaz_search_set_chain_budget(self._h, int(microseconds)), launches=0)

    def wave_counts(self):
        """(rows the last step asked for, busy trees after it).  Synchronises the stream."""
        buf = self._counts_host[0]
        self._ck(self.lib.dbaz_search_wave_counts(self._h, C.c_void_p(buf.data_ptr()), self._stream()), launches=0)
        torch.cuda.current_stream(self.device).synchronize()
        return int(buf[0]), int(buf[1])

    @property
    def priors(self):
        return self._priors[:self.n_rows]

    @property
    def values(self):
        return self._values[:self.n_rows]

    @property
    def leaf_states(self):
        return self._leaf_states[:self.n_rows]

    @property
    def leaf_kind(self):
        return self._leaf_kind[:self.n_rows]

    @property
    def planes(self):
        return self._planes[:self.n_rows]

    def set_planes(self, dtype=torch.float32, channels_last=False):
        """Choose dtype/layout of the leaf feature tensor the select kernel writes (the net's input)."""
        cfg = (dtype, bool(channels_last))
        if cfg != self._plane_cfg:
            cap = self.n_games * self.max_pending
            if channels_last:
                base = torch.zeros((cap, self.rows, self.cols, 3), dtype=dtype, device=self.device)
                self._planes = base.permute(0, 3, 1, 2)  # logical NCHW view over NHWC memory
                self._planes_base = base
            else:
                self._planes = torch.zeros((cap, 3, self.rows, self.cols), dtype=dtype, device=self.device)
                self._planes_base = self._planes
            self._plane_cfg = cfg
        return self.planes

    # ---------------------------------------------------------- state I/O
    def states_from_numpy(self, arr):
        arr = np.ascontiguousarray(arr, dtype=STATE_DTYPE).reshape(-1)
        return torch.from_numpy(arr.view(np.int64).reshape(-1, 4).copy()).to(self.device)

    @staticmethod
    def states_to_numpy(states):
        return states.detach().cpu().numpy().reshape(-1).view(STATE_DTYPE).copy()

    # ---------------------------------------------------------- game rules
    def new_states(self, n):
        """BoxesState() x n (dots_boxes_game.py:30-39)."""
        st = torch.empty((n, 4), dtype=torch.int64, device=self.device)
        self._ck(self.lib.dbaz_game_init(self._h, _ptr(st), n, self._stream()))
        return st

    def valid_moves(self, states):
        """get_valid_moves (dots_boxes_game.py:44-49) -> bool [n, A]."""
        states = self._states_arg(states)
        out = torch.empty((states.shape[0], self.A), dtype=torch.uint8, device=self.device)
        self._ck(self.lib.dbaz_game_valid_moves(self._h, _ptr(states), _ptr(out), states.shape[0], self._stream()))
        return out.bool()

    def play(self, states, moves):
        """play_ (dots_boxes_game.py:61-89) in place.  Returns (n_closed int32[n] with -1 where the
        reference raises ValueError, closed_lc int32[n, 4])."""
        states = self._states_arg(states)
        n = states.shape[0]
        moves = torch.as_tensor(moves, dtype=torch.int32, device=self.device).contiguous()
        if moves.shape != (n,):
            raise ValueError("moves must have shape [n]")
        ncl = torch.empty((n,), dtype=torch.int32, device=self.device)
        lc = torch.empty((n, 4), dtype=torch.int32, device=self.device)
        self._ck(self.lib.dbaz_game_play(self._h, _ptr(states), _ptr(moves), _ptr(ncl), _ptr(lc), n, self._stream()))
        return ncl, lc

    def result(self, states):
        """get_result (dots_boxes_game.py:51-59) -> int8 [n], RESULT_NONE (2) for None."""
        states = self._states_arg(states)
        out = torch.empty((states.shape[0],), dtype=torch.int8, device=self.device)
        self._ck(self.lib.dbaz_game_result(self._h, _ptr(states), _ptr(out), states.shape[0], self._stream()))
        return out

    def features(self, states, dtype=torch.int16, channels_last=False):
        """get_features + nn_batch_builder (dots_boxes_game.py:96-100,148-155) -> [n, 3, L+1, C+1]."""
        states = self._states_arg(states)
        n = states.shape[0]
        if channels_last:
            base = torch.empty((n, self.rows, self.cols, 3), dtype=dtype, device=self.device)
            out = base.permute(0, 3, 1, 2)
        else:
            base = out = torch.empty((n, 3, self.rows, self.cols), dtype=dtype, device=self.device)
        self._ck(self.lib.dbaz_game_features(self._h, _ptr(states), _ptr(base), _DTYPE_CODE[dtype],
                                             _capi.NHWC if channels_last else _capi.NCHW, n, self._stream()))
        return out

    def random_rollout(self, states, seed=0, game0=0, record_moves=False):
        """Uniform random legal playouts to terminal, in place.  Returns n_plies (and the move lists)."""
        states = self._states_arg(states)
        n = states.shape[0]
        plies = torch.empty((n,), dtype=torch.int32, device=self.device)
        max_plies = self.A
        moves = torch.full((n, max_plies), 255, dtype=torch.uint8, device=self.device) if record_moves else None
        self._ck(self.lib.dbaz_game_random_rollout(self._h, _ptr(states), seed, game0, _ptr(plies), _ptr(moves), max_plies,
                                                   n, self._stream()))
        return (plies, moves) if record_moves else plies

    def fake_nn(self, leaf_states, kind=0, priors=None, values=None):
        """Deterministic stand-in for the net (tests / parity runs), see include/dbaz_b200.h."""
        leaf_states = self._states_arg(leaf_states)
        n = leaf_states.shape[0]
        if priors is None:
            priors = torch.empty((n, self.A), dtype=torch.float32, device=self.device)
        if values is None:
            values = torch.empty((n,), dtype=torch.float32, device=self.device)
        self._ck(self.lib.dbaz_fake_nn(self._h, _ptr(leaf_states), _ptr(priors), _ptr(values), int(kind), n, self._stream()))
        return priors, values

    # ------------------------------------------------- leaf-eval fused stages
    def nn_stem(self, leaf_states, w01, bias_pos, k2_pos, scale, shift, out, mode=0):
        """Leaf gather + first 3x3 conv + epilogue in one kernel, from packed states (include/dbaz_b200.h).
        out: [n, L+1, C+1, cout] contiguous (NHWC), bf16/fp16."""
        n, cout = leaf_states.shape[0], out.shape[-1]
        self._ck(self.lib.dbaz_nn_stem(self._h, _ptr(leaf_states), _ptr(w01), _ptr(bias_pos), _ptr(k2_pos), _ptr(scale),
                                       _ptr(shift), _ptr(out), cout, _DTYPE_CODE[out.dtype], int(mode), n, self._stream()))
        return out

    def nn_stem_mma_pack(self, w48):
        """[48, cout] folded stem weights (bf16/fp16, contiguous) -> the fragment order nn_stem_mma() reads."""
        w48 = w48.contiguous()
        packed = torch.empty_like(w48)
        self._ck(self.lib.dbaz_nn_stem_mma_pack(self._h, _ptr(w48), _ptr(packed), w48.shape[1], self._stream()))
        return packed

    def nn_stem_mma(self, leaf_states, packed, out):
        """Leaf gather + first 3x3 conv + ReLU as one tensor-core implicit GEMM from packed states (include/dbaz_b200.h).
        packed: nn_stem_mma_pack(folded weights) in out's dtype; out: [n, L+1, C+1, cout] contiguous (NHWC), bf16/fp16."""
        n, cout = leaf_states.shape[0], out.shape[-1]
        self._ck(self.lib.dbaz_nn_stem_mma(self._h, _ptr(leaf_states), _ptr(packed), _ptr(out), cout, _DTYPE_CODE[out.dtype], n,
                                           self._stream()))
        return out

    def nn_heads(self, logits, priors=None, values=None):
        """logits [n, ld] (policy logits | value pre-activation | padding) -> softmax priors, tanh values (float32)."""
        n, ld = logits.shape
        priors = self.priors if priors is None else priors
        values = self.values if values is None else values
        self._ck(self.lib.dbaz_nn_heads(self._h, _ptr(logits), ld, _DTYPE_CODE[logits.dtype], _ptr(priors), _ptr(values), n,
                                        self._stream()))
        return priors, values

    def nn_heads_mlp(self, logits, n_hidden, v_w, priors=None, values=None):
        """logits [n, ld] (policy logits | value-head hidden pre-activations) -> softmax priors, tanh(b + relu(h) . w) with
        v_w = float32 [n_hidden + 1] (fc1's weights, then its bias)."""
        n, ld = logits.shape
        priors = self.priors if priors is None else priors
        values = self.values if values is None else values
        self._ck(self.lib.dbaz_nn_heads_mlp(self._h, _ptr(logits), ld, _DTYPE_CODE[logits.dtype], int(n_hidden), _ptr(v_w),
                                            _ptr(priors), _ptr(values), n, self._stream()))
        return priors, values

    # ------------------------------------------------- residual tower (tcgen05)
    def tower_geometry(self):
        """dict(ok, nb boards per tile, plane, tile_bytes, chunk_bytes, chunks_per_stage, channels, wp) of the fused
        residual-tower kernel for this board (include/dbaz_b200.h: dbaz_nn_tower_geometry)."""
        out = (C.c_int32 * 8)()
        self.lib.dbaz_nn_tower_geometry(self._h, out)
        keys = ("ok", "nb", "plane", "tile_bytes", "chunk_bytes", "chunks_per_stage", "channels", "wp")
        return dict(zip(keys, list(out)))

    def tower_tiles(self, n):
        """Zero-filled planar tile buffer for up to n boards (pads must stay zero: allocate once, reuse)."""
        g = self.tower_geometry()
        n_tiles = -(-int(n) // g["nb"])
        return torch.zeros((n_tiles, g["tile_bytes"]), dtype=torch.uint8, device=self.device)

    def nn_stem_mma_tiles(self, leaf_states, packed, tiles):
        """nn_stem_mma() with 64 bf16 output channels written straight into the tower's planar tiles."""
        self._ck(self.lib.dbaz_nn_stem_mma_tiles(self._h, _ptr(leaf_states), _ptr(packed), _ptr(tiles), leaf_states.shape[0], self._stream()))
        return tiles

    def tower_planarize(self, nhwc, tiles):
        """[n, L+1, C+1, 64] bf16 (contiguous NHWC) -> planar tiles, in place on `tiles`."""
        n = nhwc.shape[0]
        self._ck(self.lib.dbaz_nn_tower_planarize(self._h, _ptr(nhwc), _ptr(tiles), n, self._stream()))
        return tiles

    def tower(self, tiles, packed_w, bias, n_stages, head_cout, out):
        """The residual tower (and, with head_cout, the fused 1x1 head conv + ReLU) over the boards in `tiles`;
        out: [n, L+1, C+1, head_cout or 64] bf16 (include/dbaz_b200.h: dbaz_nn_tower)."""
        n = out.shape[0]
        self._ck(self.lib.dbaz_nn_tower(self._h, _ptr(tiles), _ptr(packed_w), _ptr(bias), int(n_stages), int(head_cout), _ptr(out), n,
                                        self._stream()))
        return out

    # ------------------------------------------- SimpleNN trunk convolution (tcgen05)
    def nn_trunk_conv_plan(self, x, y, packed_w, bias_pos, bias, pad):
        """Binds one 256-channel 3x3 convolution (zero padding `pad`) to its buffers for nn_trunk_conv (include/dbaz_b200.h:
        dbaz_nn_trunk_conv_plan).  x: [cap, hi, wi, 256] bf16 NHWC; y: [cap, ho, wo, 256] bf16; packed_w: trunk_conv_pack(w);
        bias_pos: [ho * wo, 256] and bias: [256] float32, added in that order.  Encodes the tensor maps once: build plans
        outside any stream capture."""
        cap, hi, wi, c = x.shape
        ho, wo = hi + 2 * pad - 2, wi + 2 * pad - 2
        ok = (c == 256 and x.dtype == y.dtype == packed_w.dtype == torch.bfloat16 and bias_pos.dtype == bias.dtype == torch.float32
              and tuple(y.shape) == (cap, ho, wo, 256) and tuple(packed_w.shape) == (9 * 256, 256) and tuple(bias_pos.shape) == (ho * wo, 256)
              and tuple(bias.shape) == (256,) and all(t.is_contiguous() and t.device == self.device for t in (x, y, packed_w, bias_pos, bias)))
        if not ok:
            raise ValueError("nn_trunk_conv_plan: expected contiguous bf16 x [cap, hi, wi, 256], y [cap, ho, wo, 256], "
                             "w [2304, 256] and float32 biases [ho * wo, 256], [256] on %s" % self.device)
        buf = C.create_string_buffer(int(self.lib.dbaz_nn_trunk_conv_plan_bytes()))
        self._ck(self.lib.dbaz_nn_trunk_conv_plan(self._h, _ptr(x), _ptr(y), _ptr(packed_w), _ptr(bias_pos), _ptr(bias), cap, hi, wi,
                                                  int(pad), buf), launches=0)
        return TrunkConvPlan(buf, (x, y, packed_w, bias_pos, bias))

    def nn_trunk_conv(self, plan, n):
        """Runs a planned trunk convolution for boards 0 .. n-1; returns y[:n] (rows n .. cap-1 of y are not written)."""
        self._ck(self.lib.dbaz_nn_trunk_conv(self._h, plan.buf, int(n), self._stream()))
        return plan.y[:n]

    # -------------------------------------------------------------- search
    def reset_roots(self, states=None):
        """create_root_uct_node (mcts.py:156-160) for every tree."""
        if states is None:
            states = self.new_states(self.n_games)
        states = self._states_arg(states)
        if states.shape[0] != self.n_games:
            raise ValueError("need one root state per game")
        self._noise = None
        self._ck(self.lib.dbaz_search_reset_roots(self._h, _ptr(states), self._stream()))

    def begin(self, num_reads, noise=None, coeff=0.0, pending=1):
        """Head of UCT_search (mcts.py:205-229).  num_reads: int or int32[n_games] (-1 = idle tree).
        noise: float64 [n_games, A] Dirichlet sample times legal mask, or None (alpha <= 0).
        pending: max_pending_evals, simulations in flight per tree (<= the engine's max_pending)."""
        if not 1 <= int(pending) <= self.max_pending:
            raise ValueError("pending must be in [1, %d] (Engine(max_pending=...))" % self.max_pending)
        self.pending = int(pending)
        if isinstance(num_reads, int):
            self._num_reads.fill_(num_reads)
        else:
            nr = torch.as_tensor(num_reads, dtype=torch.int32).reshape(self.n_games)
            if not (nr.is_cuda and nr.data_ptr() == self._num_reads.data_ptr()):  # a device kernel may have filled the array in place
                self._num_reads.copy_(nr, non_blocking=False)
        if noise is not None:
            noise = torch.as_tensor(noise, dtype=torch.float64).to(self.device).contiguous()
            if noise.shape != (self.n_games, self.A):
                raise ValueError("noise must have shape [n_games, A]")
        self._noise = noise
        self._ck(self.lib.dbaz_search_begin(self._h, _ptr(self._num_reads), self.pending, _ptr(noise), float(coeff), self._stream()))

    def step(self):
        """One lock-step wave: backup the leaves evaluated into self.priors/self.values, then select the
        next leaf of every tree into self.planes / self.leaf_states / self.leaf_kind."""
        dtype, cl = self._plane_cfg
        self._ck(self.lib.dbaz_search_step(self._h, _ptr(self._priors), _ptr(self._values), _ptr(self._planes_base),
                                           _DTYPE_CODE[dtype], _capi.NHWC if cl else _capi.NCHW, _ptr(self._leaf_states),
                                           _ptr(self._leaf_kind), self._stream()))
        self._nw += 1

    def step_flush(self):
        """Stop launching simulations (UCT_search's time limit) and back up the pending leaves."""
        self._ck(self.lib.dbaz_search_stop(self._h, self._stream()))
        self.step()

    def run_search(self, num_reads, evaluator, noise=None, coeff=0.0, max_reads=None, graph_waves=0, pending=1, adaptive=False):
        """UCT_search for all trees.  `evaluator(engine)` must fill engine.priors / engine.values for the
        leaves in engine.planes / engine.leaf_states, on the current stream, without host sync.

        pending: max_pending_evals (simulations in flight per tree, see begin()).
        graph_waves > 0: `graph_waves` consecutive [step kernel -> evaluator] waves are captured once in a
        CUDA graph and replayed, so the 800-wave inner loop costs one launch per `graph_waves` waves.
        Surplus waves at the end of the last replay are no-ops for trees that have finished.

        adaptive (pending == 1, graph_waves > 0): instead of a fixed number of full-width waves, the loop runs until
        no tree has work left and shrinks the evaluator's batch as trees finish -- see _run_adaptive()."""
        if adaptive and int(pending) == 1 and graph_waves > 0:
            return self._run_adaptive(num_reads, evaluator, noise, coeff, graph_waves)
        if self.compact:
            self.set_mode(False, self.max_inline)
        if max_reads is None:
            max_reads = int(num_reads) if isinstance(num_reads, int) else int(torch.as_tensor(num_reads).max())
        pending = int(pending)
        self.pending = pending
        # one wave for the expansion of an unexpanded root, one first wave of min(pending, A) simulations, then
        # `pending` per wave (terminal leaves complete inside the step and only make this an upper bound)
        first = min(pending, self.A)
        waves = 2 + max(0, -(-(max(max_reads, 0) - first) // pending))
        if graph_waves > 0:
            if noise is not None:  # a stable address for the captured step kernel
                if self._noise_buf is None:
                    self._noise_buf = torch.zeros((self.n_games, self.A), dtype=torch.float64, device=self.device)
                self._noise_buf.copy_(torch.as_tensor(noise, dtype=torch.float64).reshape(self.n_games, self.A))
                noise = self._noise_buf
            key = (id(evaluator), graph_waves, noise is not None, float(coeff), self._plane_cfg, pending, self._mode_key())
            if key not in self._graphs:
                # the evaluator is stored next to its graph: a live reference keeps id() from being recycled
                self._graphs[key] = (self._capture(evaluator, graph_waves, noise, coeff, pending), evaluator)
                self._trim_graphs()
            self.begin(num_reads, noise, coeff, pending)
            g = self._graphs[key][0]
            per_wave = 1 + int(getattr(evaluator, "engine_launches", 0))
            for _ in range((waves + graph_waves - 1) // graph_waves):
                g.replay()
                self._nl += graph_waves * per_wave
                self._nw += graph_waves
        else:
            self.begin(num_reads, noise, coeff, pending)
            for _ in range(waves):
                self.step()
                evaluator(self)
        self.step()  # flush the last backup

    # batch sizes of the adaptive loop (each one is a captured graph): n_games * k / LADDER_STEPS for k = LADDER_STEPS..1,
    # then halvings down to 64 rows
    LADDER_STEPS = 16
    ROW_MARGIN = 1.125
    UNDERSIZE = 0.9          # a batch may be this much smaller than the rows expected ...
    UNDERSIZE_GAIN = 1.05    # ... if it serves this much more rows per microsecond than the best batch that holds them
    WAVE_OVERHEAD_US = 40.0  # per-wave cost that does not depend on the batch (step kernel), for the same trade-off

    def _ladder(self, evaluator=None):
        """Evaluator batch sizes of the adaptive loop, largest first.  An evaluator whose cost is a step function of
        the batch with a known period (`batch_quantum`: the tower kernel runs boards-per-tile x SMs boards per
        wave of its persistent grid) gets rungs at whole multiples of it."""
        n, steps = self.n_games, max(1, int(self.LADDER_STEPS))
        q = int(getattr(evaluator, "batch_quantum", 0) or 0)
        if q >= 64 and n >= q:
            rows = {n} | {q * k for k in range(1, n // q + 1)}
            r = q
            while r > 64:
                r //= 2
                rows.add(max(64, -(-r // 8) * 8))
            return sorted(rows, reverse=True)
        rows = {n}
        for k in range(1, steps + 1):
            rows.add(min(n, max(64, -(-(n * k // steps) // 8) * 8)))
        r = n // steps
        while r > 64:
            r //= 2
            rows.add(min(n, max(64, -(-r // 8) * 8)))
        return sorted(rows, reverse=True)

    def _run_adaptive(self, num_reads, evaluator, noise, coeff, graph_waves):
        """The wave loop with a shrinking evaluator batch.  Leaves are handed over in compact rows (set_mode), the step
        kernel publishes how many trees still have work, and the host -- one graph replay behind the device -- picks
        the captured batch for the rows recent waves asked for (_pick_rows; never more than the busy trees; a batch
        that turns out too small only makes the surplus leaves wait a wave) and stops when no tree is busy.
        The decision for replay i+2 is taken from the counters at the end of replay i, which the host waits for:
        the schedule, and with it every evaluator batch, is reproducible."""
        self.pending = 1
        self.set_mode(True, self.max_inline)
        if noise is not None:
            if self._noise_buf is None:
                self._noise_buf = torch.zeros((self.n_games, self.A), dtype=torch.float64, device=self.device)
            self._noise_buf.copy_(torch.as_tensor(noise, dtype=torch.float64).reshape(self.n_games, self.A))
            noise = self._noise_buf
        ladder = self._ladder(evaluator)
        per_wave = 1 + int(getattr(evaluator, "engine_launches", 0))
        graphs = self._ladder_graphs(evaluator, graph_waves, noise, coeff)
        if self.device_loop:
            try:
                return self._run_device_loop(num_reads, evaluator, noise, coeff, graphs)
            except EngineError as exc:  # a driver that cannot build the conditional graph: the host-driven loop does the same
                import warnings
                warnings.warn("device-driven wave loop unavailable (%s); using the host-driven loop" % exc)
                self.device_loop = False
        self.begin(num_reads, noise, coeff, 1)
        stream = torch.cuda.current_stream(self.device)
        events = []
        busy = self.wave_counts()[1]  # trees that take part in this search (begin() counted them)
        if busy == 0:
            return
        rows, i = min(r for r in ladder if r >= busy), 0
        self.last_schedule = []  # (evaluator batch, busy trees it was chosen for) per replay, for profiling
        while True:
            self.last_schedule.append((rows, busy))
            graphs[rows].replay()
            self._count_replay(graphs[rows])
            slot = self._counts_host[i % self._counts_host.shape[0]]
            self.lib.dbaz_search_wave_counts(self._h, C.c_void_p(slot.data_ptr()), self._stream())
            ev = torch.cuda.Event()
            ev.record(stream)
            events.append((ev, slot))
            i += 1
            if len(events) >= 2:
                ev0, slot0 = events.pop(0)
                ev0.synchronize()
                busy = int(slot0[1])
                if busy == 0:
                    break
                # the evaluator's next batch: what the waves of that replay asked for at most, plus a margin, never
                # more than the busy trees.  Too small is safe (set_batch_rows: the surplus leaves wait a wave).
                want = min(busy, int(int(slot0[2]) * self.ROW_MARGIN) + 32)
                rows = self._pick_rows(ladder, want, id(evaluator))

    def _run_device_loop(self, num_reads, evaluator, noise, coeff, graphs):
        """The adaptive loop as ONE graph launch (include/dbaz_b200.h: dbaz_search_loop_build): a WHILE node around a
        SWITCH over the captured rung graphs and a decision kernel; the host neither reads counters nor waits."""
        key = id(graphs)
        if key not in self._loops:
            ladder = sorted(graphs, reverse=True)
            n = len(ladder)
            raws = (C.c_uint64 * n)(*[int(graphs[r].raw_cuda_graph()) for r in ladder])
            rows = (C.c_int32 * n)(*ladder)
            us = (C.c_float * n)(*[float(self._eval_us.get((id(evaluator), r), 0.0)) for r in ladder])
            out = C.c_uint64()
            rc = self.lib.dbaz_search_loop_build(self._h, raws, rows, us, n, 1 << 16, float(self.ROW_MARGIN), float(self.UNDERSIZE),
                                                 float(self.UNDERSIZE_GAIN), float(self.WAVE_OVERHEAD_US), C.byref(out))
            if rc != 0:
                raise EngineError(self.lib.dbaz_last_error(self._h).decode())
            self._loops[key] = (out.value, ladder, graphs)
        loop, ladder, _ = self._loops[key]
        self.begin(num_reads, noise, coeff, 1)
        self._ck(self.lib.dbaz_search_loop_launch(self._h, C.c_uint64(loop), self._stream()), launches=0)
        if self._loop_counts_host is None:
            self._loop_counts_host = torch.zeros((32, 48), dtype=torch.int32).pin_memory()
            self._loop_slot = 0
        if len(self._loop_pending) >= self._loop_counts_host.shape[0] - 1:
            self._fold_loop_counts()  # the ring of pinned slots is about to wrap
        counts = self._loop_counts_host[self._loop_slot % self._loop_counts_host.shape[0]][:len(ladder)]
        self._loop_slot += 1
        self.lib.dbaz_search_loop_counts(self._h, C.c_uint64(loop), C.c_void_p(counts.data_ptr()), self._stream())
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.device))
        self._loop_pending.append((ev, counts, ladder, graphs))
        self.last_schedule = None

    def _ladder_graphs(self, evaluator, graph_waves, noise, coeff, short_tail=True):
        """{batch rows: CUDA graph of `graph_waves` [step -> evaluator] waves} for every rung of the ladder (compact mode).
        Every batch size is captured up front: capturing re-binds the search head and idles all trees."""
        key = (id(evaluator), graph_waves, noise is not None, float(coeff), self._plane_cfg, 1, self._mode_key(), "ladder", self.LADDER_STEPS,
               short_tail, tuple(self._ladder(evaluator)))
        if key not in self._graphs:
            graphs = {}
            for rows in self._ladder(evaluator):
                self._batch_rows = rows
                try:
                    graphs[rows] = self._capture(evaluator, self._rung_waves(rows, graph_waves) if short_tail else graph_waves, noise, coeff, 1)
                finally:
                    self._batch_rows = None
            self._graphs[key] = (graphs, evaluator)
            self._trim_graphs()
        return self._graphs[key][0]

    def _rung_waves(self, rows, graph_waves):
        """Waves per graph replay of a rung: the small rungs run at the end of a search, where the host's decision lag
        (two replays) is pure overhead once the last tree has finished, so their graphs are shorter."""
        return max(1, graph_waves // 4) if rows * 8 <= self.n_games else graph_waves

    def _pick_rows(self, ladder, want, ev_id):
        """The batch size for waves that are expected to ask for `want` rows: the rung that holds them and serves the most
        rows per microsecond of evaluator time -- or a rung up to 10 % short of `want` when that is clearly cheaper per row
        served (library GEMM/conv kernels are step functions of the batch: a rung just past a tile-wave boundary costs a
        whole extra wave).  A short rung is allowed because the surplus leaves simply wait a wave
        (dbaz_search_set_batch_rows); it has to win by UNDERSIZE_GAIN because those leaves' trees fall a wave behind."""
        def score(r):
            us = self._eval_us.get((ev_id, r))
            return None if us is None else min(r, want) / (us + self.WAVE_OVERHEAD_US)
        fit = [r for r in ladder if r >= want] or [ladder[0]]
        scored = [(score(r), r) for r in fit]
        if any(sc is None for sc, _ in scored):
            return min(fit)
        best_sc, best = max(scored)
        for r in ladder:
            if self.UNDERSIZE * want <= r < want:
                sc = score(r)
                if sc is not None and sc > best_sc * self.UNDERSIZE_GAIN:
                    best_sc, best = sc / self.UNDERSIZE_GAIN * 1.0001, r  # a further short rung must beat this one outright
        return best

    def _count_replay(self, g):
        launches, waves = self._graph_cost.get(id(g), (0, 0))
        self._nl += launches
        self._nw += waves

    MAX_GRAPH_SETS = 6

    def _trim_graphs(self):
        """Captured graphs (and the evaluators they keep alive) of configurations not used for a while are dropped,
        oldest first: a coach loop builds a new evaluator every generation."""
        while len(self._graphs) > self.MAX_GRAPH_SETS:
            old = self._graphs.pop(next(iter(self._graphs)))[0]
            loop = self._loops.pop(id(old), None)
            if loop is not None:
                torch.cuda.synchronize(self.device)
                self._fold_loop_counts()
                self.lib.dbaz_search_loop_destroy(self._h, C.c_uint64(loop[0]))

    CHAIN_COUNT_CAP = 64   # with a time budget the count only stops runaway chains

    def _mode_key(self):
        return (self.compact, self.max_inline, self.eval_cache_log2, self.chain_us)

    def _capture(self, evaluator, graph_waves, noise, coeff, pending=1):
        # warm up the evaluator alone (allocator, cuDNN heuristics); no leaf is pending between searches,
        # so overwriting priors/values here is harmless
        cur = torch.cuda.current_stream(self.device)
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            for _ in range(3):
                evaluator(self)
        cur.wait_stream(side)
        torch.cuda.synchronize(self.device)
        if self._graph_pool is None:
            self._graph_pool = torch.cuda.graph_pool_handle()  # graphs never run concurrently and keep nothing alive
        if self._batch_rows is not None:
            # what this batch size costs on the device (a graph of 4 calls, so that no launch overhead is in the figure):
            # the adaptive loop weighs rows served against time (see _pick_rows)
            g0 = torch.cuda.CUDAGraph()  # private pool: dies with the graph
            with torch.cuda.graph(g0):
                for _ in range(4):
                    evaluator(self)
            g0.replay()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            g0.replay()
            g0.replay()
            b.record()
            torch.cuda.synchronize(self.device)
            self._eval_us[(id(evaluator), self._batch_rows)] = a.elapsed_time(b) * 125.0
            del g0
        # the captured step kernels carry the noise pointer / coeff of begin() and the evaluator's batch; bind them first
        self._noise = noise
        self.lib.dbaz_search_set_batch_rows(self._h, int(self._batch_rows or 0))
        # small batches are the tail of a search, where a wave costs the evaluator's latency floor whatever it serves:
        # longer in-kernel chains there save whole waves (any bound gives the same results)
        inline = self.max_inline
        factor = 1
        if self._batch_rows is not None and inline > 0:
            factor = 4 if self._batch_rows * 16 <= self.n_games else (2 if self._batch_rows * 4 <= self.n_games else 1)
        budget = int(self.chain_us) * factor if (inline > 0 and int(pending) == 1) else 0
        inline = self.CHAIN_COUNT_CAP if budget > 0 else inline * factor
        self.lib.dbaz_search_set_mode(self._h, 1 if self.compact else 0, int(inline))
        self._ck(self.lib.dbaz_search_set_chain_budget(self._h, budget), launches=0)
        self.lib.dbaz_search_begin(self._h, _ptr(self._idle_reads), int(pending), _ptr(noise), float(coeff), self._stream())
        g = torch.cuda.CUDAGraph(keep_graph=True) if self._batch_rows is not None else torch.cuda.CUDAGraph()
        n0, w0 = self._nl, self._nw
        with torch.cuda.graph(g, pool=self._graph_pool):
            for _ in range(graph_waves):
                self.step()
                evaluator(self)
        self._graph_cost[id(g)] = (self._nl - n0, self._nw - w0)  # engine kernels / waves one replay stands for
        self._nl, self._nw = n0, w0  # capture enqueues nothing
        self.lib.dbaz_search_set_batch_rows(self._h, 0)
        self.lib.dbaz_search_set_mode(self._h, 1 if self.compact else 0, int(self.max_inline))
        self.lib.dbaz_search_set_chain_budget(self._h, 0)
        return g

    def root_visits(self):
        out = torch.empty((self.n_games, self.A), dtype=torch.int32, device=self.device)
        self._ck(self.lib.dbaz_search_root_visits(self._h, _ptr(out), self._stream()))
        return out

    def root_children(self):
        """(W float32, priors float64, sign int32, ucb float64), each [n_games, A]."""
        n, A = self.n_games, self.A
        W = torch.empty((n, A), dtype=torch.float32, device=self.device)
        P = torch.empty((n, A), dtype=torch.float64, device=self.device)
        S = torch.empty((n, A), dtype=torch.int32, device=self.device)
        U = torch.empty((n, A), dtype=torch.float64, device=self.device)
        self._ck(self.lib.dbaz_search_root_children(self._h, _ptr(W), _ptr(P), _ptr(S), _ptr(U), self._stream()))
        return W, P, S, U

    def tree_stats(self):
        """(stats int32[n, 8] = root_N, max_deepness, tree_size, terminal_count, is_expanded, is_terminal,
        n_nodes, error; root_W float32[n]; q float32[n])."""
        n = self.n_games
        st = torch.empty((n, 8), dtype=torch.int32, device=self.device)
        W = torch.empty((n,), dtype=torch.float32, device=self.device)
        q = torch.empty((n,), dtype=torch.float32, device=self.device)
        self._ck(self.lib.dbaz_search_tree_stats(self._h, _ptr(st), _ptr(W), _ptr(q), self._stream()))
        return st, W, q

    def root_states(self):
        out = torch.empty((self.n_games, 4), dtype=torch.int64, device=self.device)
        self._ck(self.lib.dbaz_search_root_states(self._h, _ptr(out), self._stream()))
        return out

    def node_view(self, tree, node):
        """dict of one node of one tree (include/dbaz_b200.h: dbaz_search_node), host values.  Synchronises."""
        A, dev = self.A, self.device
        st = torch.zeros((1, 4), dtype=torch.int64, device=dev)
        W = torch.zeros((A,), dtype=torch.float32, device=dev)
        N = torch.zeros((A,), dtype=torch.int32, device=dev)
        P = torch.zeros((A,), dtype=torch.float64, device=dev)
        ch = torch.zeros((A,), dtype=torch.int32, device=dev)
        sg = torch.zeros((A,), dtype=torch.int32, device=dev)
        U = torch.zeros((A,), dtype=torch.float64, device=dev)
        own = torch.zeros((8,), dtype=torch.int32, device=dev)
        oW = torch.zeros((1,), dtype=torch.float32, device=dev)
        self._ck(self.lib.dbaz_search_node(self._h, int(tree), int(node), _ptr(st), _ptr(W), _ptr(N), _ptr(P), _ptr(ch), _ptr(sg), _ptr(U),
                                           _ptr(own), _ptr(oW), self._stream()))
        own = own.cpu().numpy()
        if own[7]:
            raise IndexError("tree %d has no node %d" % (tree, node))
        return {"state": self.states_to_numpy(st)[0], "W": W.cpu().numpy(), "visits": N.cpu().numpy(), "priors": P.cpu().numpy(),
                "child": ch.cpu().numpy(), "sign": sg.cpu().numpy(), "ucb": U.cpu().numpy(), "N": int(own[0]), "is_expanded": bool(own[1]),
                "is_terminal": bool(own[2]), "parent": int(own[3]), "parent_action": int(own[4]), "depth": int(own[5]),
                "n_nodes": int(own[6]), "own_W": np.float32(oW.cpu().numpy()[0])}

    def tree_busy(self):
        """bool[n_games]: the tree's search is still running."""
        out = torch.empty((self.n_games,), dtype=torch.int8, device=self.device)
        self._ck(self.lib.dbaz_search_tree_busy(self._h, _ptr(out), self._stream()))
        return out.bool()

    def selfplay_pick(self, bufs):
        """get_next_move + the sample of play_game (self_play.py:27-74) for every tree whose search has finished
        (include/dbaz_b200.h: dbaz_selfplay_pick); bufs: _capi.SelfplayBuffers of device pointers."""
        self._ck(self.lib.dbaz_selfplay_pick(self._h, C.byref(bufs), self._stream()))

    def selfplay_restart(self, bufs, first=False):
        """After advance_roots(bufs.moves): budget and noise row of the games that go on (dbaz_selfplay_restart)."""
        self._ck(self.lib.dbaz_selfplay_restart(self._h, C.byref(bufs), 1 if first else 0, self._stream()))

    def advance_roots(self, moves, reuse=True):
        """init_mcts_tree (mcts.py:163-180) for every tree; moves int32[n_games], -1 = keep."""
        moves = torch.as_tensor(moves, dtype=torch.int32).to(self.device).contiguous()
        if moves.shape != (self.n_games,):
            raise ValueError("moves must have shape [n_games]")
        self._noise = None
        self._ck(self.lib.dbaz_search_advance_roots(self._h, _ptr(moves), 1 if reuse else 0, self._stream()))

    def status(self):
        """Synchronises.  Returns dict(errors, sims, path_nodes, max_nodes_used); raises if a tree faulted."""
        out = (C.c_int64 * 8)()
        rc = self.lib.dbaz_search_status(self._h, out, self._stream())
        d = {"errors": out[0], "sims": out[1], "path_nodes": out[2], "max_nodes_used": out[3], "terminal_leaves": out[4],
             "cache_hits": out[5]}
        if rc != 0:
            raise EngineError(self.lib.dbaz_last_error(self._h).decode())
        return d


class FakeNetEvaluator:
    """Evaluator for parity runs: the deterministic fake net, on device."""

    engine_launches = 1  # one k_fake_nn per wave

    def __init__(self, kind=0):
        self.kind = kind

    def __call__(self, eng):
        eng.fake_nn(eng.leaf_states, self.kind, eng.priors, eng.values)
