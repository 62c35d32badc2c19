"""Root-PUCT search over tensor state batches -- call-compatible mirror of the reference's
``v1/python/mcts_gpu.py`` (``GpuStateBatch`` :40-145, ``V1RootMCTSConfig`` :223-236, ``RootSearchBatchOutput``
:250-259, ``V1RootMCTS.search_batch`` :1249-1457), running on the liuzhou_b200 kernels.

Semantics kept from the reference (SURVEY.md Appendix A): every root child is evaluated once, values are moved to
the parent's perspective only when the side to move changes, terminal children are overridden by
``+-tanh(k * material / 18)``, N visits are allocated by fp32 PUCT with fixed leaf values, the policy target is
``visits^(1/T)``, moves are sampled from the log-space stable policy.  RNG draws (Gamma noise [R,M], multinomial
[R,M], forced-uniform multinomial) come from torch's generator in the reference's order, so identical seeds give
identical draws.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional, Tuple

import torch

from . import v0_core
from .net import InferenceNet, bucket_logits_to_scalar

PLACEMENT_DIM, MOVEMENT_DIM, SELECTION_DIM, AUXILIARY_DIM = 36, 144, 36, 4
TOTAL_ACTION_DIM = 220
MAX_MOVE_COUNT = 144
NO_CAPTURE_DRAW_LIMIT = 36
LOSE_PIECE_THRESHOLD = 4
PHASE_MOVEMENT, PHASE_CAPTURE_SELECTION, PHASE_COUNTER_REMOVAL = 4, 5, 7

_FIELDS = ("board", "marks_black", "marks_white", "phase", "current_player", "pending_marks_required",
           "pending_marks_remaining", "pending_captures_required", "pending_captures_remaining",
           "forced_removals_done", "move_count", "moves_since_capture")


@dataclass
class GpuStateBatch:
    """Tensor-native game state batch (reference tensor layout, 12 tensors)."""

    board: torch.Tensor
    marks_black: torch.Tensor
    marks_white: torch.Tensor
    phase: torch.Tensor
    current_player: torch.Tensor
    pending_marks_required: torch.Tensor
    pending_marks_remaining: torch.Tensor
    pending_captures_required: torch.Tensor
    pending_captures_remaining: torch.Tensor
    forced_removals_done: torch.Tensor
    move_count: torch.Tensor
    moves_since_capture: torch.Tensor

    @property
    def device(self) -> torch.device:
        return self.board.device

    @property
    def batch_size(self) -> int:
        return int(self.board.shape[0])

    def tensors(self) -> Tuple[torch.Tensor, ...]:
        return tuple(getattr(self, f) for f in _FIELDS)

    def to(self, device) -> "GpuStateBatch":
        return GpuStateBatch(*(t.to(torch.device(device)) for t in self.tensors()))

    def slice(self, index: int) -> "GpuStateBatch":
        return GpuStateBatch(*(t[index:index + 1] for t in self.tensors()))

    def select(self, indices) -> "GpuStateBatch":
        if isinstance(indices, list):
            if not indices:
                raise ValueError("indices must not be empty.")
            idx = torch.tensor(indices, dtype=torch.int64, device=self.device)
        else:
            idx = indices.to(device=self.device, dtype=torch.int64).view(-1)
            if int(idx.numel()) == 0:
                raise ValueError("indices must not be empty.")
        return GpuStateBatch(*(t.index_select(0, idx) for t in self.tensors()))

    @staticmethod
    def initial(device, batch_size: int = 1) -> "GpuStateBatch":
        dev = torch.device(device)
        z = lambda: torch.zeros((batch_size,), dtype=torch.int64, device=dev)  # noqa: E731
        return GpuStateBatch(
            board=torch.zeros((batch_size, 6, 6), dtype=torch.int8, device=dev),
            marks_black=torch.zeros((batch_size, 6, 6), dtype=torch.bool, device=dev),
            marks_white=torch.zeros((batch_size, 6, 6), dtype=torch.bool, device=dev),
            phase=torch.ones((batch_size,), dtype=torch.int64, device=dev),
            current_player=torch.ones((batch_size,), dtype=torch.int64, device=dev),
            pending_marks_required=z(), pending_marks_remaining=z(), pending_captures_required=z(),
            pending_captures_remaining=z(), forced_removals_done=z(), move_count=z(), moves_since_capture=z())


def states_to_model_input(batch: GpuStateBatch) -> torch.Tensor:
    return v0_core.states_to_model_input(batch.board, batch.marks_black, batch.marks_white, batch.phase,
                                         batch.current_player)


def encode_actions_fast(batch: GpuStateBatch):
    return v0_core.encode_actions_fast(*batch.tensors()[:10], PLACEMENT_DIM, MOVEMENT_DIM, SELECTION_DIM,
                                       AUXILIARY_DIM)


def batch_apply_moves_compat(batch: GpuStateBatch, action_codes: torch.Tensor,
                             parent_indices: torch.Tensor) -> GpuStateBatch:
    out = v0_core.batch_apply_moves(*batch.tensors(), action_codes.to(device=batch.device, dtype=torch.int32),
                                    parent_indices.to(device=batch.device, dtype=torch.int64))
    return GpuStateBatch(*out)


@dataclass
class V1RootMCTSConfig:
    num_simulations: int = 128
    exploration_weight: float = 1.0
    temperature: float = 1.0
    add_dirichlet_noise: bool = True
    dirichlet_alpha: float = 0.3
    dirichlet_epsilon: float = 0.25
    sample_moves: bool = True
    autocast_dtype: str = "bfloat16"       # reference default is float16 (mcts_gpu.py:232); B200 path is bf16
    child_eval_mode: str = "value_only"
    soft_value_k: float = 2.0
    sparse_ply: int = 1                    # the experimental multi-ply mode (declared unsafe upstream) is not offered
    sparse_top_k: int = 8


@dataclass
class RootSearchBatchOutput:
    model_input: torch.Tensor
    legal_mask: torch.Tensor
    policy_dense: torch.Tensor
    root_value: torch.Tensor
    terminal_mask: torch.Tensor
    chosen_action_indices: torch.Tensor
    chosen_action_codes: torch.Tensor
    chosen_valid_mask: torch.Tensor


class V1RootMCTS:
    """Root-only PUCT search (depth 1) with every op on the GPU."""

    def __init__(self, model, config: V1RootMCTSConfig, device, inference_engine=None, collect_timing: bool = False):
        self.config = config
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("liuzhou_b200.V1RootMCTS runs on CUDA devices only (no CPU fallback)")
        if int(config.sparse_ply) > 1:
            raise RuntimeError("sparse_ply > 1 is not supported (upstream marks it unsafe); use the tree backend")
        self.model = model
        dt = str(config.autocast_dtype).strip().lower()
        dtype = torch.float16 if dt in ("fp16", "float16", "half") else torch.bfloat16
        self.net = model if isinstance(model, InferenceNet) else InferenceNet(model, self.device, dtype)
        self._terminal_soft_override_count = 0
        self._forced_uniform_pick_count = 0

    # -- network -------------------------------------------------------------------------------------
    def _forward_model(self, inputs_f32: torch.Tensor):
        return self.net.forward(inputs_f32)

    def _evaluate_batch(self, batch: GpuStateBatch):
        inputs = states_to_model_input(batch)
        log_p1, log_p2, log_pmc, raw_values = self._forward_model(inputs)
        values = bucket_logits_to_scalar(raw_values).float()
        legal_mask, metadata = encode_actions_fast(batch)
        probs, _ = v0_core.project_policy_logits_fast(log_p1, log_p2, log_pmc, legal_mask, PLACEMENT_DIM, MOVEMENT_DIM,
                                                      SELECTION_DIM, AUXILIARY_DIM)
        return inputs, legal_mask, metadata, probs.float(), values

    def _evaluate_values_only(self, batch: GpuStateBatch) -> torch.Tensor:
        _p1, _p2, _pm, raw_values = self._forward_model(states_to_model_input(batch))
        return bucket_logits_to_scalar(raw_values).float()

    # -- helpers with the reference's semantics ----------------------------------------------------------
    @staticmethod
    def _terminal_mask_from_next_state(batch: GpuStateBatch) -> torch.Tensor:     # mcts_gpu.py:658-675
        post = batch.phase.eq(PHASE_MOVEMENT) | batch.phase.eq(PHASE_CAPTURE_SELECTION) | batch.phase.eq(PHASE_COUNTER_REMOVAL)
        black = batch.board.eq(1).sum(dim=(1, 2))
        white = batch.board.eq(-1).sum(dim=(1, 2))
        win = post & (black.lt(LOSE_PIECE_THRESHOLD) | white.lt(LOSE_PIECE_THRESHOLD))
        draw = batch.move_count.ge(MAX_MOVE_COUNT) | batch.moves_since_capture.ge(NO_CAPTURE_DRAW_LIMIT)
        return win | draw

    @staticmethod
    def _soft_tanh_from_board_black(board: torch.Tensor, soft_value_k: float) -> torch.Tensor:   # :677-686
        black = board.eq(1).sum(dim=(1, 2)).to(torch.float32)
        white = board.eq(-1).sum(dim=(1, 2)).to(torch.float32)
        return torch.tanh((black - white) / 18.0 * float(soft_value_k))

    @staticmethod
    def _child_values_to_parent_perspective(child_values, parent_players, child_players):        # :688-708
        vals = child_values.to(torch.float32).view(-1)
        same = child_players.to(torch.int64).view(-1).eq(parent_players.to(torch.int64).view(-1))
        return torch.where(same, vals, -vals)

    @staticmethod
    def _normalize_temperatures(temperatures, batch_size, default_temperature, device):
        if temperatures is None:
            return torch.full((batch_size,), float(default_temperature), dtype=torch.float32, device=device)
        if isinstance(temperatures, (float, int)):
            return torch.full((batch_size,), float(temperatures), dtype=torch.float32, device=device)
        t = torch.as_tensor(temperatures, dtype=torch.float32, device=device).view(-1)
        if int(t.numel()) != batch_size:
            raise ValueError(f"temperatures size mismatch: expected {batch_size}, got {int(t.numel())}")
        return t

    @staticmethod
    def _stable_legal_policy_from_visits(*, visits, valid_mask, root_temps):                      # :853-898
        mask_f = valid_mask.to(torch.float32)
        safe_visits = torch.nan_to_num(visits.to(torch.float32), nan=0.0, posinf=0.0, neginf=0.0).clamp_min(1e-8)
        safe_temps = torch.nan_to_num(root_temps.to(torch.float32), nan=1.0, posinf=1.0, neginf=1.0).clamp_min(1e-6).view(-1, 1)
        logits = (torch.log(safe_visits) / safe_temps).masked_fill(~valid_mask, float("-inf"))
        row_max = logits.max(dim=1, keepdim=True).values
        row_max = torch.where(torch.isfinite(row_max), row_max, torch.zeros_like(row_max))
        exp_logits = torch.nan_to_num(torch.exp(logits - row_max) * mask_f, nan=0.0, posinf=0.0, neginf=0.0)
        row_sum = exp_logits.sum(dim=1, keepdim=True)
        fallback = mask_f / mask_f.sum(dim=1, keepdim=True).clamp_min(1.0)
        no_valid = mask_f.sum(dim=1).eq(0.0)
        fallback[no_valid, 0] = 1.0
        probs = exp_logits / row_sum.clamp_min(1e-8)
        bad = torch.logical_or(~torch.isfinite(row_sum.view(-1)), row_sum.view(-1).le(0.0))
        probs = torch.where(bad.view(-1, 1), fallback, probs) * mask_f
        probs = probs / probs.sum(dim=1, keepdim=True).clamp_min(1e-8)
        return torch.nan_to_num(probs, nan=0.0, posinf=0.0, neginf=0.0)

    def get_timing(self, reset: bool = False):
        return {"timing_ms": {}, "timing_calls": {},
                "counters": {"terminal_soft_override_count": int(self._terminal_soft_override_count),
                             "forced_uniform_pick_count": int(self._forced_uniform_pick_count)}}

    # -- the search ------------------------------------------------------------------------------------
    @torch.no_grad()
    def search_batch(self, state: GpuStateBatch, *, temperatures=None, add_dirichlet_noise: Optional[bool] = None,
                     force_uniform_random_mask: Optional[torch.Tensor] = None) -> RootSearchBatchOutput:
        cfg = self.config
        batch_size = int(state.batch_size)
        dev = state.device
        add_noise = cfg.add_dirichlet_noise if add_dirichlet_noise is None else bool(add_dirichlet_noise)
        force_uniform_mask = None
        if force_uniform_random_mask is not None:
            force_uniform_mask = torch.as_tensor(force_uniform_random_mask, device=dev).to(torch.bool).view(-1)
            if int(force_uniform_mask.numel()) != batch_size:
                raise ValueError("force_uniform_random_mask size mismatch")
        temp_values = self._normalize_temperatures(temperatures, batch_size, cfg.temperature, dev)

        model_input, legal_mask, metadata, probs, values = self._evaluate_batch(state)
        root_values = values.clone().to(torch.float32)
        policy_dense = torch.zeros((batch_size, TOTAL_ACTION_DIM), dtype=torch.float32, device=dev)
        chosen_action_indices = torch.full((batch_size,), -1, dtype=torch.int64, device=dev)
        chosen_action_codes = torch.full((batch_size, 4), -1, dtype=torch.int32, device=dev)
        chosen_valid_mask = torch.zeros((batch_size,), dtype=torch.bool, device=dev)

        (terminal_mask, valid_root_indices, counts, valid_mask, legal_index_mat, priors_mat, action_code_mat,
         flat_indices, action_codes_all, parent_indices_all) = v0_core.root_pack_sparse_actions(legal_mask, probs, metadata)

        if int(valid_root_indices.numel()) > 0:
            num_roots, max_actions = int(valid_root_indices.numel()), int(valid_mask.shape[1])
            if add_noise and max_actions > 1:                                          # :1329-1339
                eps, alpha = float(cfg.dirichlet_epsilon), float(cfg.dirichlet_alpha)
                alpha_t = torch.full_like(priors_mat, alpha, dtype=torch.float32)
                noise = torch.distributions.Gamma(alpha_t, torch.ones_like(priors_mat)).sample() * valid_mask.to(torch.float32)
                noise = noise / noise.sum(dim=1, keepdim=True).clamp_min(1e-8)
                mixed = (1.0 - eps) * priors_mat + eps * noise
                priors_mat = torch.where(counts.gt(1).view(-1, 1), mixed, priors_mat)

            child_batch = batch_apply_moves_compat(state, action_codes_all, parent_indices_all)
            child_values = self._evaluate_values_only(child_batch)
            parent_player = state.current_player.index_select(0, parent_indices_all)
            child_leaf_values = self._child_values_to_parent_perspective(child_values, parent_player,
                                                                         child_batch.current_player)
            terminal_child = self._terminal_mask_from_next_state(child_batch)
            soft_from_black = self._soft_tanh_from_board_black(child_batch.board, float(cfg.soft_value_k))
            parent_sign = torch.where(parent_player.ge(0), 1.0, -1.0).to(torch.float32)
            child_leaf_values = torch.where(terminal_child, soft_from_black * parent_sign, child_leaf_values)

            leaf_mat = torch.zeros((num_roots, max_actions), dtype=torch.float32, device=dev)
            leaf_mat.view(-1).index_copy_(0, flat_indices, child_leaf_values)

            visits, value_sum, _ = v0_core.root_puct_allocate_visits(priors_mat, leaf_mat, valid_mask,
                                                                     max(1, int(cfg.num_simulations)),
                                                                     float(cfg.exploration_weight))
            root_temps = temp_values.index_select(0, valid_root_indices)
            (policy_dense, chosen_action_indices, chosen_action_codes, chosen_valid_mask,
             root_value_vec) = v0_core.root_finalize_from_visits(legal_index_mat, action_code_mat, valid_mask, visits,
                                                                 value_sum, valid_root_indices, batch_size,
                                                                 TOTAL_ACTION_DIM, root_temps, False)
            if bool(cfg.sample_moves and max_actions > 1):                             # :1410-1424
                legal_policy = self._stable_legal_policy_from_visits(visits=visits, valid_mask=valid_mask,
                                                                     root_temps=root_temps)
                picks = torch.multinomial(legal_policy, num_samples=1).view(-1)
                chosen_action_indices.index_copy_(0, valid_root_indices, legal_index_mat.gather(1, picks.view(-1, 1)).view(-1))
                chosen_action_codes.index_copy_(
                    0, valid_root_indices, action_code_mat.gather(1, picks.view(-1, 1, 1).expand(-1, 1, 4)).view(-1, 4))
            if force_uniform_mask is not None and bool(force_uniform_mask.any().item()):   # :1425-1445
                force_local_idx = torch.where(force_uniform_mask.index_select(0, valid_root_indices))[0]
                if int(force_local_idx.numel()) > 0:
                    fvm = valid_mask.index_select(0, force_local_idx).to(torch.float32)
                    fpicks = torch.multinomial(fvm / fvm.sum(dim=1, keepdim=True).clamp_min(1e-8), num_samples=1).view(-1)
                    f_idx = legal_index_mat.index_select(0, force_local_idx).gather(1, fpicks.view(-1, 1)).view(-1)
                    f_codes = action_code_mat.index_select(0, force_local_idx).gather(
                        1, fpicks.view(-1, 1, 1).expand(-1, 1, 4)).view(-1, 4)
                    f_roots = valid_root_indices.index_select(0, force_local_idx)
                    chosen_action_indices.index_copy_(0, f_roots, f_idx)
                    chosen_action_codes.index_copy_(0, f_roots, f_codes)
                    chosen_valid_mask.index_fill_(0, f_roots, True)
                    self._forced_uniform_pick_count += int(force_local_idx.numel())
            root_values.index_copy_(0, valid_root_indices, root_value_vec)

        return RootSearchBatchOutput(model_input=model_input, legal_mask=legal_mask.to(torch.bool),
                                     policy_dense=policy_dense, root_value=root_values, terminal_mask=terminal_mask,
                                     chosen_action_indices=chosen_action_indices,
                                     chosen_action_codes=chosen_action_codes, chosen_valid_mask=chosen_valid_mask)
