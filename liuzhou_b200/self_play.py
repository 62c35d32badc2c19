"""Wave-batched self-play entry -- call-compatible with the reference's ``self_play_v1_gpu``
(v1/python/self_play_gpu_runner.py:21-307): same arguments, same ``(TensorSelfPlayBatch, SelfPlayV1Stats)`` result,
same trajectory format and schedule (per-game temperature switch at ``temperature_threshold`` plies, forced-uniform
opening, Dirichlet noise every ply, no refill of finished games inside a wave).

``search_backend``:
  "root"  reference production semantics (root-PUCT over all children, V1RootMCTS.search_batch);
  "tree"  full MCTS on the device tree (select / expand / backup kernels), the search north_star asks for; mirrors
          the reference's portable self-play (v1/python/portable_cpp_self_play.py): subtree reuse after every move
          (``tree_reuse``), policy target temperature / prior pseudocount (``policy_target_*``, tree backend only).
"""
from __future__ import annotations

import time
from dataclasses import dataclass, field
from typing import Any, Dict, Optional, Tuple

import torch

from . import native, v0_core
from .mcts_gpu import TOTAL_ACTION_DIM, GpuStateBatch, V1RootMCTS, V1RootMCTSConfig
from .net import InferenceNet
from .compact import expand_rows_fixed
from .trajectory_buffer import TensorSelfPlayBatch, TensorTrajectoryBuffer
from .tree_search import TreeMCTS

_PIECE_DELTA_MIN, _PIECE_DELTA_MAX = -18, 18


@dataclass
class SelfPlayV1Stats:
    """v1/python/self_play_types.py:11-53."""

    num_games: int
    num_positions: int
    black_wins: int
    white_wins: int
    draws: int
    avg_game_length: float
    elapsed_sec: float
    positions_per_sec: float
    games_per_sec: float
    step_timing_ms: Dict[str, float] = field(default_factory=dict)
    step_timing_ratio: Dict[str, float] = field(default_factory=dict)
    step_timing_calls: Dict[str, int] = field(default_factory=dict)
    mcts_counters: Dict[str, int] = field(default_factory=dict)
    piece_delta_buckets: Dict[str, int] = field(default_factory=dict)
    policy_target_audit: Dict[str, Any] = field(default_factory=dict)
    device: str = ""
    fallback_count: int = 0
    fallback_reasons: Tuple[str, ...] = ()

    def to_dict(self) -> Dict[str, object]:
        d: Dict[str, object] = {k: float(getattr(self, k)) for k in (
            "num_games", "num_positions", "black_wins", "white_wins", "draws", "avg_game_length", "elapsed_sec",
            "positions_per_sec", "games_per_sec")}
        d["step_timing_ms"] = {k: float(v) for k, v in self.step_timing_ms.items()}
        d["step_timing_ratio"] = {k: float(v) for k, v in self.step_timing_ratio.items()}
        d["step_timing_calls"] = {k: int(v) for k, v in self.step_timing_calls.items()}
        d["mcts_counters"] = {k: int(v) for k, v in self.mcts_counters.items()}
        d["piece_delta_buckets"] = {k: int(v) for k, v in self.piece_delta_buckets.items()}
        d["policy_target_audit"] = dict(self.policy_target_audit or {})
        d["device"] = str(self.device)
        d["fallback_count"] = int(self.fallback_count)
        d["fallback_reasons"] = list(self.fallback_reasons)
        return d


def _soft_tanh_from_board_black(board: torch.Tensor, k: float) -> torch.Tensor:
    black = board.eq(1).sum(dim=(1, 2)).to(torch.float32)
    white = board.eq(-1).sum(dim=(1, 2)).to(torch.float32)
    return torch.tanh((black - white) / 18.0 * float(k))


def _popcount36(x: torch.Tensor) -> torch.Tensor:
    from .engine import _popcount36 as pc

    return pc(x)


@dataclass
class TreePlyRules:
    """Per-game schedule of a tree-backend self-play ply (the settings of ``self_play_v1_gpu(search_backend="tree")``)."""

    temperature_init: float
    temperature_final: float
    temperature_threshold: int
    add_dirichlet_noise: bool
    sample_moves: bool
    opening_random_n: int
    max_plies: int
    soft_value_k: float


@dataclass
class TreePly:
    """What one ply did.  ``states`` / ``plies`` are the values after the moves; ``result`` / ``soft`` (from black's
    perspective) are meaningful where ``newly`` (the game ended this ply)."""

    out: object                      # TreeSearchOutput
    chosen: torch.Tensor             # int64[G] action played (< 0: none)
    legal_words: torch.Tensor        # int64[G,4] encode_actions_fast legal bits of the states before the move
    sign: torch.Tensor               # int8[G] +1 black / -1 white to move before the move
    states: torch.Tensor
    plies: torch.Tensor
    move: torch.Tensor               # bool[G] a move was applied
    newly: torch.Tensor              # bool[G] the game ended this ply
    result: torch.Tensor             # f32[G]
    soft: torch.Tensor               # f32[G]


def tree_ply(tree_mcts: TreeMCTS, states: torch.Tensor, plies: torch.Tensor, active: torch.Tensor, rules: TreePlyRules,
             *, live_rows: Optional[int] = None, restart_states: Optional[torch.Tensor] = None) -> TreePly:
    """One ply of every active game on the packed layout, without a host synchronisation: the search (and its RNG draws),
    the legal rows, the forced-uniform opening picks, the step / finish rules of module.cpp:632-871, result and soft
    value, and the subtree-reuse advance.  The one implementation of these rules: the wave loop of
    ``self_play_v1_gpu(search_backend="tree")`` and ``SelfPlayActor`` both call it.

    ``live_rows``: a host-side upper bound of the active games; the simulation waves then evaluate only the live trees'
    leaves (``TreeMCTS.set_live``).  ``restart_states`` int64[G,4]: the games that end this ply start again from these
    states in the tree (``TreeMCTS.advance`` restart path); None leaves their trees as they are."""
    mask36 = (1 << 36) - 1
    if live_rows is not None:
        tree_mcts.set_live(active)
    temps = torch.where(plies < int(rules.temperature_threshold), float(rules.temperature_init),
                        float(rules.temperature_final)).to(torch.float32)
    out = tree_mcts.search(states, active=active, temperatures=temps, add_dirichlet_noise=rules.add_dirichlet_noise,
                           sample_moves=rules.sample_moves, live_rows=live_rows)
    if live_rows is not None:
        tree_mcts.warm_buckets()         # first compacted search of this engine: capture the smaller wave batches once
    chosen = out.chosen_action_indices
    # legal-mask rows as the reference stores them: v0_core.encode_actions_fast semantics (no game-over check)
    legal_words = native.legal_masks(states, scalar_semantics=False)[0]
    if rules.opening_random_n > 0:
        force = (plies < rules.opening_random_n) & ~out.terminal_mask & active
        lm = native.mask_words_to_bool(legal_words).to(torch.float32)
        tot = lm.sum(dim=1, keepdim=True)
        uni = torch.where(tot > 0, lm / tot.clamp_min(1.0), torch.full_like(lm, 1.0 / TOTAL_ACTION_DIM))
        chosen = torch.where(force, torch.multinomial(uni, 1).view(-1), chosen)
    white_to_move = (states[:, 0] >> 39) & 1                           # meta bit 3 of w0 >> 36
    sign_now = (1 - 2 * white_to_move).to(torch.int8)
    # self_play_step_inplace (module.cpp:632-871) on the packed layout
    immediate = active & out.terminal_mask                            # no legal action: the side to move loses
    move = active & ~out.terminal_mask
    nxt = native.apply_actions(states, chosen.clamp_min(0).to(torch.int32))
    states = torch.where(move.view(-1, 1), nxt, states).contiguous()
    plies = plies + move.to(torch.int32)
    w0, w1 = states[:, 0], states[:, 1]
    meta = (w0 >> 36) & 0xFFFFFFF
    phase = meta & 7
    black, white = _popcount36(w0 & mask36), _popcount36(w1 & mask36)
    post = (phase == 4) | (phase == 5) | (phase == 7)
    winner = torch.where(post & (white < 4), 1, torch.where(post & (black < 4), -1, 0))     # :817-824
    draw = (((meta >> 14) & 255) >= 144) | (((meta >> 22) & 63) >= 36)
    fin = move & ((winner != 0) | draw | (plies >= int(rules.max_plies)))
    newly = immediate | fin
    res_now = torch.where(immediate, -sign_now.to(torch.float32), winner.to(torch.float32))
    soft_now = torch.tanh((black - white).to(torch.float32) / 18.0 * float(rules.soft_value_k))
    # subtree reuse (portable_cpp_self_play.py:170): the played child becomes the root; finished games keep -1
    keep = torch.where(move & ~fin, chosen, torch.full_like(chosen, -1))
    if restart_states is None:
        tree_mcts.advance(keep)
    else:
        tree_mcts.advance(keep, restart_states, newly)
    return TreePly(out=out, chosen=chosen, legal_words=legal_words, sign=sign_now, states=states, plies=plies, move=move,
                   newly=newly, result=res_now, soft=soft_now)


def _play_wave_tree(actor, rules: TreePlyRules, progress: Optional[list] = None):
    """One wave of ``actor.num_games`` games from the initial position to the end of every game, with the reference's
    wave semantics (self_play_gpu_runner.py:159-256: every live game appends one row per ply, no refill, step / finalise
    rules of module.cpp:632-871): the actor (``SelfPlayActor``) with ``finish()`` before its first step, so no host round
    trip per ply and the live-game count read every 4 plies (the simulation waves evaluate only the live trees' leaves).
    -> (rows int64[n, 42] in the reference's append order -- ply-major, live games ascending --, game records, stats).
    ``progress`` (optional list) receives (ply, live-game upper bound, time) at every live-game count."""
    g, max_plies = actor.num_games, int(rules.max_plies)
    actor.rules = rules
    actor._allocate(max_plies, g * max_plies)        # every game of the wave fits the output
    actor.reset()
    actor.finish()
    while not actor.idle:
        actor.step()
        if progress is not None and actor._finish_plies % 4 == 0:
            progress.append((actor._finish_plies, actor._live_upper, time.perf_counter()))
    rows, _, rec, stats = actor._take_output()
    n = int(rows.shape[0])
    # emission order (game by game) -> ply-major, slot ascending
    game = torch.repeat_interleave(torch.arange(rec.shape[0], device=rows.device), rec[:, 2], output_size=n)
    ply = torch.arange(n, device=rows.device) - rec[:, 3].index_select(0, game)
    order = torch.argsort(ply * g + rec[:, 1].index_select(0, game))
    return rows.index_select(0, order), rec, stats


def self_play_v1_gpu(
    model,
    num_games: int,
    mcts_simulations: int,
    temperature_init: float,
    temperature_final: float,
    temperature_threshold: int,
    exploration_weight: float,
    device: str,
    add_dirichlet_noise: bool = True,
    dirichlet_alpha: float = 0.3,
    dirichlet_epsilon: float = 0.25,
    soft_value_k: float = 2.0,
    opening_random_moves: int = 0,
    max_game_plies: int = 512,
    sample_moves: bool = True,
    concurrent_games: int = 8,
    child_eval_mode: str = "value_only",
    sparse_ply: int = 1,
    sparse_top_k: int = 8,
    inference_engine=None,
    collect_step_timing: bool = False,
    verbose: bool = False,
    search_backend: str = "root",
    leaves_per_wave: int = 1,
    tree_reuse: bool = True,
    policy_target_temperature: Optional[float] = None,
    policy_target_prior_pseudocount: float = 0.0,
    engine_cache: Optional[Dict[Any, Any]] = None,
) -> Tuple[TensorSelfPlayBatch, SelfPlayV1Stats]:
    """``engine_cache`` (optional dict owned by the caller, e.g. one per worker): the search engines built for this call
    (device tree arenas, captured CUDA graphs) are kept there and reused by later calls with the same shape / settings
    instead of being rebuilt per call."""
    if num_games <= 0:
        raise ValueError("num_games must be positive.")
    dev = torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError("liuzhou_b200.self_play_v1_gpu runs on CUDA devices only (no CPU fallback)")
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    if search_backend not in ("root", "tree"):
        raise ValueError("search_backend must be 'root' or 'tree'")
    max_plies = max(1, int(max_game_plies))
    opening_random_n = max(0, int(opening_random_moves))
    wave_size = max(1, min(int(concurrent_games), int(num_games)))
    sims = max(1, int(mcts_simulations))
    net = model if isinstance(model, InferenceNet) else InferenceNet(model, dev)

    root_mcts = tree_mcts = None
    if search_backend == "root":
        root_mcts = V1RootMCTS(net, V1RootMCTSConfig(
            num_simulations=sims, exploration_weight=float(exploration_weight), temperature=float(temperature_init),
            add_dirichlet_noise=bool(add_dirichlet_noise), dirichlet_alpha=float(dirichlet_alpha),
            dirichlet_epsilon=float(dirichlet_epsilon), sample_moves=bool(sample_moves),
            child_eval_mode=str(child_eval_mode), soft_value_k=float(soft_value_k), sparse_ply=int(sparse_ply),
            sparse_top_k=int(sparse_top_k)), dev)

    outcome_counts = torch.zeros((3,), dtype=torch.int64, device=dev)
    piece_delta_hist = torch.zeros((_PIECE_DELTA_MAX - _PIECE_DELTA_MIN + 1,), dtype=torch.int64, device=dev)
    game_lengths = torch.zeros((int(num_games),), dtype=torch.int64, device=dev)
    started = time.perf_counter()
    evals = 0

    if search_backend == "tree":
        from .actor import SelfPlayActor

        parts, actor = [], None
        for wave_base in range(0, int(num_games), wave_size):
            wave_games = min(wave_size, int(num_games) - wave_base)
            cache_key = ("tree", id(net), wave_games, sims, float(exploration_weight), bool(add_dirichlet_noise),
                         float(dirichlet_alpha), float(dirichlet_epsilon), bool(sample_moves), int(leaves_per_wave),
                         bool(tree_reuse), policy_target_temperature, float(policy_target_prior_pseudocount))
            if engine_cache is not None and cache_key in engine_cache:
                actor = engine_cache[cache_key]
            if actor is None or actor.num_games != wave_games:
                actor = SelfPlayActor(
                    net, wave_games, device=dev, mcts_simulations=sims, exploration_weight=float(exploration_weight),
                    add_dirichlet_noise=bool(add_dirichlet_noise), dirichlet_alpha=float(dirichlet_alpha),
                    dirichlet_epsilon=float(dirichlet_epsilon), sample_moves=bool(sample_moves),
                    leaves_per_wave=int(leaves_per_wave), tree_reuse=bool(tree_reuse),
                    policy_target_temperature=policy_target_temperature,
                    policy_target_prior_pseudocount=float(policy_target_prior_pseudocount), max_game_plies=max_plies,
                    output_capacity=wave_games * max_plies)
                if engine_cache is not None:
                    engine_cache[cache_key] = actor
            rows, rec, wave_stats = _play_wave_tree(actor, TreePlyRules(
                temperature_init=float(temperature_init), temperature_final=float(temperature_final),
                temperature_threshold=int(temperature_threshold), add_dirichlet_noise=bool(add_dirichlet_noise),
                sample_moves=bool(sample_moves), opening_random_n=opening_random_n, max_plies=max_plies,
                soft_value_k=float(soft_value_k)))
            parts.append(rows)
            game_lengths.index_copy_(0, rec[:, 1] + wave_base, rec[:, 2])
            outcome_counts += torch.tensor([wave_stats.black_wins, wave_stats.white_wins, wave_stats.draws],
                                           dtype=torch.int64, device=dev)
            piece_delta_hist += torch.tensor([wave_stats.piece_delta_buckets[str(d)]
                                              for d in range(_PIECE_DELTA_MIN, _PIECE_DELTA_MAX + 1)],
                                             dtype=torch.int64, device=dev)
            if verbose:
                oc = outcome_counts.tolist()
                print(f"[v1.self_play] games={min(wave_base + wave_games, num_games)}/{num_games} "
                      f"W/L/D={oc[0]}/{oc[1]}/{oc[2]}")
        batch = expand_rows_fixed(parts[0] if len(parts) == 1 else torch.cat(parts), check=False)
        tree_mcts = actor.mcts
        buffer = None
    else:
        buffer = TensorTrajectoryBuffer(dev, TOTAL_ACTION_DIM, max_steps_hint=min(max_plies, 160),
                                        concurrent_games_hint=min(wave_size, num_games))

    for wave_base in (range(0, int(num_games), wave_size) if search_backend == "root" else ()):
        wave_games = min(wave_size, int(num_games) - wave_base)
        states = GpuStateBatch.initial(dev, batch_size=wave_games)
        step_index_matrix = torch.full((wave_games, max_plies), -1, dtype=torch.int64, device=dev)
        step_counts = torch.zeros((wave_games,), dtype=torch.int64, device=dev)
        plies = torch.zeros((wave_games,), dtype=torch.int64, device=dev)
        done = torch.zeros((wave_games,), dtype=torch.bool, device=dev)

        while True:
            active_idx = torch.where(~done)[0]
            n_active = int(active_idx.numel())
            if n_active == 0:
                break
            active_plies = plies.index_select(0, active_idx)
            active_states = states.select(active_idx)
            temps = torch.where(active_plies < int(temperature_threshold), float(temperature_init),
                                float(temperature_final)).to(torch.float32)
            force_uniform = active_plies < opening_random_n if opening_random_n > 0 else None
            search = root_mcts.search_batch(active_states, temperatures=temps,
                                            add_dirichlet_noise=add_dirichlet_noise,
                                            force_uniform_random_mask=force_uniform)
            model_input, legal_mask, policy_dense = search.model_input, search.legal_mask, search.policy_dense
            player_sign = active_states.current_player
            chosen_codes, terminal_mask, chosen_valid = (search.chosen_action_codes, search.terminal_mask,
                                                         search.chosen_valid_mask)

            step_indices = buffer.append_steps(model_input=model_input, legal_mask=legal_mask,
                                               policy_dense=policy_dense, player_sign=player_sign)
            step_positions = step_counts.index_select(0, active_idx)
            step_index_matrix[active_idx, step_positions] = step_indices
            step_counts.index_add_(0, active_idx, torch.ones((n_active,), dtype=torch.int64, device=dev))
            finalize_slots, result_local, soft_local = v0_core.self_play_step_inplace(
                *states.tensors(), plies, done, active_idx, chosen_codes, terminal_mask, chosen_valid, int(max_plies),
                float(soft_value_k))
            if int(finalize_slots.numel()) > 0:
                final_boards = states.board.index_select(0, finalize_slots)
                delta = (final_boards.eq(1).sum(dim=(1, 2)) - final_boards.eq(-1).sum(dim=(1, 2))).to(torch.int64)
                piece_delta_hist.add_(torch.bincount(torch.clamp(delta - _PIECE_DELTA_MIN, 0, piece_delta_hist.numel() - 1),
                                                     minlength=piece_delta_hist.numel()))
                soft_local = _soft_tanh_from_board_black(final_boards, float(soft_value_k))
                fin_slots, fin_lengths, outcome_delta = buffer.finalize_games_inplace(
                    step_index_matrix=step_index_matrix, step_counts=step_counts, slots=finalize_slots,
                    result_from_black=result_local, soft_value_from_black=soft_local)
                if int(fin_slots.numel()) > 0:
                    game_lengths.index_copy_(0, fin_slots + int(wave_base), fin_lengths)
                outcome_counts.add_(outcome_delta)
        if verbose:
            oc = outcome_counts.tolist()
            print(f"[v1.self_play] games={min(wave_base + wave_games, num_games)}/{num_games} W/L/D={oc[0]}/{oc[1]}/{oc[2]}")

    torch.cuda.synchronize(dev)
    elapsed = max(1e-9, time.perf_counter() - started)
    if buffer is not None:
        batch = buffer.build()
    oc = outcome_counts.tolist()
    hist = piece_delta_hist.cpu().tolist()
    if tree_mcts is not None:
        evals = tree_mcts.evals
    counters = {"network_evals": int(evals)}
    if root_mcts is not None:
        counters.update(root_mcts.get_timing()["counters"])
    keys = ("root_puct_ms", "pack_writeback_ms", "self_play_step_ms", "finalize_ms")
    stats = SelfPlayV1Stats(
        num_games=int(num_games), num_positions=batch.num_samples, black_wins=int(oc[0]), white_wins=int(oc[1]),
        draws=int(oc[2]), avg_game_length=float(game_lengths.to(torch.float32).mean().item()), elapsed_sec=elapsed,
        positions_per_sec=float(batch.num_samples / elapsed), games_per_sec=float(num_games / elapsed),
        step_timing_ms={k: 0.0 for k in keys}, step_timing_ratio={k: 0.0 for k in keys},
        step_timing_calls={k: 0 for k in keys}, mcts_counters=counters,
        piece_delta_buckets={str(d): int(hist[d - _PIECE_DELTA_MIN]) for d in range(_PIECE_DELTA_MIN, _PIECE_DELTA_MAX + 1)},
        device=str(dev))
    return batch, stats
