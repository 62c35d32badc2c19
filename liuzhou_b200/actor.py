"""Refilling self-play actor: G concurrent games on the device tree search that keeps its batch full, finalises every
finished game's rows with the outcome and hands them out, and picks up new weights between plies.

    actor = SelfPlayActor(net, 4096, device="cuda", mcts_simulations=200)
    while training:
        actor.step(plies=8)                 # no host synchronisation
        games = actor.drain()               # one host synchronisation
        trainer.add(games.batch)            # reference-format TensorSelfPlayBatch, value targets final
        actor.load_state_dict(new_weights)  # games in flight continue on the new weights

Per ply: the rules of ``self_play.tree_ply`` (the same function the wave loop of ``self_play_v1_gpu(search_backend=
"tree")`` runs), then two kernels (csrc/lz_actor.cu): ``lzb_actor_record`` writes every live game's row, in the
336-byte fixed format of ``compact.compact_rows_fixed``, into a per-slot arena; ``lzb_actor_emit`` appends the rows of
the games that ended (value targets filled in), their action traces and one record per game to a linear output, in
ascending slot order within a ply.  A finished slot restarts from the initial position at once.  ``finish()`` stops
the refill: the games in flight play out with the wave loop's live-game compaction and ``idle`` becomes true.
"""
from __future__ import annotations

import ctypes
import time
from dataclasses import dataclass
from typing import Optional

import torch

from . import native
from ._lib import check, i64, lib, ptr, stream_ptr
from .compact import FIXED_ROW_WORDS, expand_rows_fixed
from .net import InferenceNet
from .self_play import _PIECE_DELTA_MAX, _PIECE_DELTA_MIN, SelfPlayV1Stats, TreePlyRules, tree_ply
from .trajectory_buffer import TensorSelfPlayBatch
from .tree_search import TreeMCTS, TreeMCTSConfig

ROW_BYTES = FIXED_ROW_WORDS * 8
RECORD_WORDS = 8
_CTL_WORDS = 48                  # see include/liuzhou_b200.h, lzb_actor_record / lzb_actor_emit
_CTL_ROWS, _CTL_GAMES, _CTL_SERIAL, _CTL_OVERFLOW, _CTL_ROW_FLAGS = 0, 1, 2, 3, 4
_CTL_OUTCOMES, _CTL_DELTA = 6, 9


def arena_bytes(num_games: int, max_game_plies: int) -> int:
    """Device memory of the per-slot game arenas: one fixed row, one int8 sign and one int16 action per (slot, ply),
    plus an int32 row count per slot."""
    return int(num_games) * int(max_game_plies) * (ROW_BYTES + 1 + 2) + 4 * int(num_games)


def output_bytes(output_capacity: int) -> int:
    """Device memory of the output buffer: per row a fixed row and an int16 action, per game (at most one per row) a
    record of RECORD_WORDS int64."""
    return int(output_capacity) * (ROW_BYTES + 2 + 8 * RECORD_WORDS)


@dataclass
class ActorGames:
    """Finished games of one ``drain()``, in emission order (the ply they ended, then slot ascending).  Game i owns rows
    ``row_offset[i] .. row_offset[i] + length[i] - 1`` of ``batch`` / ``rows`` / ``actions``, in ply order."""

    batch: TensorSelfPlayBatch       # reference format, value targets final
    rows: torch.Tensor               # int64[n, 42] the same rows in the fixed 336-byte format
    actions: torch.Tensor            # int16[n] action played from each row's position (-1: none, the side to move lost)
    serial: torch.Tensor             # int64[games] per-actor game number, in order of emission
    slot: torch.Tensor               # int64[games]
    length: torch.Tensor             # int64[games] rows of the game
    row_offset: torch.Tensor         # int64[games]
    finish_step: torch.Tensor        # int64[games] actor step (ply count since construction) in which the game ended
    piece_delta: torch.Tensor        # int64[games] black - white pieces at the end
    result: torch.Tensor             # f32[games] from black's perspective: +1, -1, 0
    soft_value: torch.Tensor         # f32[games] tanh(k (black - white) / 18) at the end
    stats: SelfPlayV1Stats


class SelfPlayActor:
    """``model_or_net``: a ChessNet or an InferenceNet.  The search settings mean what they mean for
    ``self_play_v1_gpu(search_backend="tree")``; temperatures and the random opening follow each game's own ply count.
    ``output_capacity``: rows the output holds between two drains (default 64 per slot).  Games that do not fit are
    not written, and the next ``drain()`` discards the output and raises; the actor itself stays usable."""

    def __init__(self, model_or_net, num_games: int, *, device, mcts_simulations: int = 200,
                 temperature_init: float = 1.0, temperature_final: float = 0.1, temperature_threshold: int = 10,
                 exploration_weight: float = 1.0, add_dirichlet_noise: bool = True, dirichlet_alpha: float = 0.3,
                 dirichlet_epsilon: float = 0.25, soft_value_k: float = 2.0, opening_random_moves: int = 0,
                 max_game_plies: int = 512, sample_moves: bool = True, tree_reuse: bool = True,
                 leaves_per_wave: int = 1, policy_target_temperature: Optional[float] = None,
                 policy_target_prior_pseudocount: float = 0.0, output_capacity: Optional[int] = None):
        g, max_plies = int(num_games), int(max_game_plies)
        if g <= 0:
            raise ValueError("num_games must be positive")
        if max_plies <= 0:
            raise ValueError("max_game_plies must be positive")
        if int(mcts_simulations) <= 0 or int(leaves_per_wave) <= 0:
            raise ValueError("mcts_simulations and leaves_per_wave must be positive")
        cap = 64 * g if output_capacity is None else int(output_capacity)
        if cap < max_plies:
            raise ValueError("output_capacity must hold at least one game of max_game_plies rows")
        dev = torch.device(device)
        if dev.type != "cuda":
            raise RuntimeError("liuzhou_b200.SelfPlayActor runs on CUDA devices only (no CPU fallback)")
        if dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        self.device, self.num_games = dev, g
        self.net = model_or_net if isinstance(model_or_net, InferenceNet) else InferenceNet(model_or_net, dev)
        self.mcts = TreeMCTS(self.net, g, TreeMCTSConfig(
            num_simulations=int(mcts_simulations), exploration_weight=float(exploration_weight),
            add_dirichlet_noise=bool(add_dirichlet_noise), dirichlet_alpha=float(dirichlet_alpha),
            dirichlet_epsilon=float(dirichlet_epsilon), sample_moves=bool(sample_moves),
            leaves_per_wave=int(leaves_per_wave), reuse_subtree=bool(tree_reuse),
            policy_target_temperature=policy_target_temperature,
            policy_target_prior_pseudocount=float(policy_target_prior_pseudocount)), dev)
        self.rules = TreePlyRules(
            temperature_init=float(temperature_init), temperature_final=float(temperature_final),
            temperature_threshold=int(temperature_threshold), add_dirichlet_noise=bool(add_dirichlet_noise),
            sample_moves=bool(sample_moves), opening_random_n=max(0, int(opening_random_moves)), max_plies=max_plies,
            soft_value_k=float(soft_value_k))
        self._initial = native.init_states(g, dev)
        self._all = torch.ones((g,), dtype=torch.bool, device=dev)
        self._nrows = torch.zeros((g,), dtype=torch.int32, device=dev)
        self._ctl = torch.zeros((_CTL_WORDS,), dtype=torch.int64, device=dev)
        self.max_game_plies = self.output_capacity = 0
        self._allocate(max_plies, cap)
        self.steps = 0
        self._evals_at_drain = 0
        self._drained_at = time.perf_counter()
        self.reset()

    def _allocate(self, max_plies: int, capacity: int) -> None:
        """(Re)size the per-slot game arenas (row (slot, ply) = slot * max_plies + ply) and the linear output."""
        g, dev = self.num_games, self.device
        if max_plies != self.max_game_plies:
            self._arena = torch.empty((g * max_plies, FIXED_ROW_WORDS), dtype=torch.int64, device=dev)
            self._signs = torch.empty((g * max_plies,), dtype=torch.int8, device=dev)
            self._actions = torch.empty((g * max_plies,), dtype=torch.int16, device=dev)
            self.max_game_plies = max_plies
        if capacity != self.output_capacity:
            self._out_rows = torch.empty((capacity, FIXED_ROW_WORDS), dtype=torch.int64, device=dev)
            self._out_actions = torch.empty((capacity,), dtype=torch.int16, device=dev)
            self._records = torch.empty((capacity, RECORD_WORDS), dtype=torch.int64, device=dev)
            self.output_capacity = capacity

    def reset(self) -> None:
        """Start a new game in every slot and empty the output (the game serials run on).  ``finish()`` is undone."""
        g, dev = self.num_games, self.device
        self.states = self._initial.clone()
        self.plies = torch.zeros((g,), dtype=torch.int32, device=dev)
        self.done = torch.zeros((g,), dtype=torch.bool, device=dev)
        self._nrows.zero_()
        self._ctl[_CTL_ROWS:_CTL_GAMES + 1].zero_()
        self._ctl[_CTL_OUTCOMES:].zero_()
        self.mcts.set_live(None)
        self.mcts._advanced = False                  # the next search starts from reset roots
        self.finishing = False
        self.idle = False
        self._finish_plies = 0
        self._live_upper = g

    # ---- the two kernels ---------------------------------------------------------------------------------------------
    # bool tensors are passed as they are: torch stores a bool as one byte holding 0 or 1, the kernels' uint8 layout
    def _record(self, states: torch.Tensor, active: torch.Tensor, policy: torch.Tensor, chosen: torch.Tensor) -> None:
        if active.dtype != torch.bool or policy.dtype != torch.float32 or chosen.dtype != torch.int64:
            raise TypeError("active must be bool, policy float32 and chosen int64")
        act, pol, ch = active.contiguous(), policy.contiguous(), chosen.contiguous()
        check(lib().lzb_actor_record(ptr(states), ptr(act), ptr(pol), ptr(ch), i64(self.num_games),
                                     ctypes.c_int32(self.max_game_plies), ptr(self._nrows), ptr(self._arena),
                                     ptr(self._signs), ptr(self._actions), ptr(self._ctl), stream_ptr(self.device)))

    def _emit(self, finished: torch.Tensor, result: torch.Tensor, soft: torch.Tensor, states: torch.Tensor) -> None:
        if finished.dtype != torch.bool or result.dtype != torch.float32 or soft.dtype != torch.float32:
            raise TypeError("finished must be bool, result and soft float32")
        fin, res, sv = finished.contiguous(), result.contiguous(), soft.contiguous()
        check(lib().lzb_actor_emit(ptr(fin), ptr(res), ptr(sv), ptr(states), i64(self.num_games),
                                   ctypes.c_int32(self.max_game_plies), ptr(self._nrows), ptr(self._arena),
                                   ptr(self._signs), ptr(self._actions), ptr(self._out_rows), ptr(self._out_actions),
                                   ptr(self._records), i64(self.output_capacity), ptr(self._ctl), i64(self.steps),
                                   stream_ptr(self.device)))

    # ---- public API --------------------------------------------------------------------------------------------------
    @torch.no_grad()
    def step(self, plies: int = 1) -> None:
        """Play ``plies`` plies of every live game.  While refilling there is no host synchronisation; after ``finish()``
        the host reads the live-game count every 4 plies, as the wave loop does."""
        with torch.cuda.device(self.device):
            for _ in range(int(plies)):
                if self.idle:
                    return
                self._ply()

    def _ply(self) -> None:
        live_rows = None
        if self.finishing:
            if self._finish_plies > 0 and self._finish_plies % 4 == 0:
                self._live_upper = int((~self.done).sum().item())
                if self._live_upper == 0:
                    self.idle = True
                    self.mcts.set_live(None)
                    return
            live_rows = self._live_upper
            active = ~self.done
        else:
            active = self._all
        before = self.states
        p = tree_ply(self.mcts, before, self.plies, active, self.rules, live_rows=live_rows,
                     restart_states=None if self.finishing else self._initial)
        self._record(before, active, p.out.policy_dense, p.chosen)
        self._emit(p.newly, p.result, p.soft, p.states)
        if self.finishing:
            self.states, self.plies = p.states, p.plies
            self.done = self.done | p.newly
            self._finish_plies += 1
        else:
            self.states = torch.where(p.newly.view(-1, 1), self._initial, p.states).contiguous()
            self.plies = torch.where(p.newly, torch.zeros_like(p.plies), p.plies)
        self.steps += 1

    def finish(self) -> None:
        """Stop refilling: finished slots stay empty, the games in flight play out, then ``idle`` is true."""
        if not self.finishing:
            self.finishing = True
            self._finish_plies = 0
            self._live_upper = self.num_games

    def load_state_dict(self, state_dict) -> None:
        """New network weights (``InferenceNet.load_state_dict``), in stream order between two plies: the games in flight
        continue on them, the captured search graphs stay valid."""
        self.net.load_state_dict(state_dict)

    def _take_output(self):
        """-> (rows, actions, records, stats) of the games emitted since the last drain, and empties the output; one host
        read.  Raises on overflow (after emptying the output) or on a sticky error flag."""
        with torch.cuda.device(self.device):
            snap = torch.cat([self._ctl, self.mcts.tree.counters[1:2].to(torch.int64)]).cpu().tolist()
            now = time.perf_counter()
            n, games = int(snap[_CTL_ROWS]), int(snap[_CTL_GAMES])
            if snap[_CTL_OVERFLOW] & 2:
                raise RuntimeError("SelfPlayActor game arena overflow: a game recorded more than max_game_plies rows")
            if snap[_CTL_ROW_FLAGS]:
                raise RuntimeError("SelfPlayActor emitted rows that are not representable in the fixed-row format")
            self.mcts.tree._raise_flags(int(snap[_CTL_WORDS]))
            rows = self._out_rows[:n].clone() if n <= self.output_capacity else None
            actions = self._out_actions[:n].clone() if rows is not None else None
            rec = self._records[:games].clone() if rows is not None else None
            outcomes = snap[_CTL_OUTCOMES:_CTL_OUTCOMES + 3]
            hist = snap[_CTL_DELTA:_CTL_DELTA + _PIECE_DELTA_MAX - _PIECE_DELTA_MIN + 1]
            evals = self.mcts.evals - self._evals_at_drain
            elapsed = max(1e-9, now - self._drained_at)
            # empty the output (cursors, overflow flag, per-drain statistics); the serial counter runs on
            self._ctl[_CTL_ROWS:_CTL_GAMES + 1].zero_()
            self._ctl[_CTL_OVERFLOW] = 0
            self._ctl[_CTL_OUTCOMES:].zero_()
            self._evals_at_drain = self.mcts.evals
            self._drained_at = now
            if snap[_CTL_OVERFLOW] & 1:
                raise RuntimeError(f"SelfPlayActor output overflow: {games} games ({n} rows) finished since the last drain, "
                                   f"more than the {self.output_capacity} rows of the output; they are discarded. Drain "
                                   "more often or raise output_capacity; the actor can go on")
        keys = ("root_puct_ms", "pack_writeback_ms", "self_play_step_ms", "finalize_ms")
        stats = SelfPlayV1Stats(
            num_games=games, num_positions=n, black_wins=int(outcomes[0]), white_wins=int(outcomes[1]),
            draws=int(outcomes[2]), avg_game_length=float(n / games) if games else 0.0, elapsed_sec=elapsed,
            positions_per_sec=float(n / elapsed), games_per_sec=float(games / elapsed),
            step_timing_ms={k: 0.0 for k in keys}, step_timing_ratio={k: 0.0 for k in keys},
            step_timing_calls={k: 0 for k in keys}, mcts_counters={"network_evals": int(evals)},
            piece_delta_buckets={str(d): int(hist[d - _PIECE_DELTA_MIN])
                                 for d in range(_PIECE_DELTA_MIN, _PIECE_DELTA_MAX + 1)},
            device=str(self.device))
        return rows, actions, rec, stats

    def drain(self) -> ActorGames:
        """The games finished since the last drain, in emission order; one host synchronisation.  Raises if the output
        overflowed (its games are then discarded and the actor goes on with an empty output), a row was not
        representable, or the tree search set a sticky error flag."""
        rows, actions, rec, stats = self._take_output()
        with torch.cuda.device(self.device):
            batch = expand_rows_fixed(rows, check=False)
            vs = rec[:, 6:7].contiguous().view(torch.float32)
        return ActorGames(batch=batch, rows=rows, actions=actions, serial=rec[:, 0], slot=rec[:, 1], length=rec[:, 2],
                          row_offset=rec[:, 3], finish_step=rec[:, 4], piece_delta=rec[:, 5], result=vs[:, 0].clone(),
                          soft_value=vs[:, 1].clone(), stats=stats)


__all__ = ["SelfPlayActor", "ActorGames", "arena_bytes", "output_bytes"]
