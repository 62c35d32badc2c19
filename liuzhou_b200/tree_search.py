"""Batched full-tree MCTS search on one GPU: the device tree (tree.py / csrc/lz_tree.cu) + the bf16 network
(net.py) + the fused head kernel, with one simulation wave captured in a CUDA graph.

Host-side counterpart of the reference's ``PortableCppMCTS.search_batch`` (v1/python/portable_cpp_mcts.py:243-390):
prepare_roots -> evaluate -> expand roots -> optional Dirichlet noise on root priors -> S x (select leaves ->
evaluate -> expand + backup) -> root outputs -> policy from visit counts.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional

import torch

from .net import InferenceNet
from .tree import ACTION_DIM, DeviceTreeBatch, encode_inputs, heads_to_priors


@dataclass
class TreeMCTSConfig:
    num_simulations: int = 200
    exploration_weight: float = 1.0
    temperature: float = 1.0
    add_dirichlet_noise: bool = True
    dirichlet_alpha: float = 0.3
    dirichlet_epsilon: float = 0.25
    sample_moves: bool = True
    leaves_per_wave: int = 1          # K = 1 reproduces the reference's visit counts exactly
    virtual_loss: float = 1.0
    nodes_per_tree_hint: Optional[int] = None
    use_cuda_graph: bool = True
    # keep the played child's subtree between consecutive searches of a game (``advance()`` after every move), as the
    # reference's portable self-play does (portable_cpp_self_play.py:170, portable_mcts.cpp:739-768)
    reuse_subtree: bool = False
    # policy TARGET (what the trajectory stores) = softmax(log(N + beta * P) / T_target); None keeps the legacy
    # behaviour of reusing the per-game action-selection temperature (portable_cpp_mcts.py:340-354, train.py:2838-2856)
    policy_target_temperature: Optional[float] = None
    policy_target_prior_pseudocount: float = 0.0


@dataclass
class TreeSearchOutput:
    legal_mask: torch.Tensor          # bool[T,220]  (children of each root)
    visit_counts: torch.Tensor        # int32[T,220]
    policy_dense: torch.Tensor        # f32[T,220]   policy target: (N + beta P)^(1/T_target) normalised
    selection_policy_dense: torch.Tensor  # f32[T,220] move-selection policy: N^(1/T) normalised (one-hot for T <= 1e-6)
    root_value: torch.Tensor          # f32[T]
    root_action_values: torch.Tensor  # f32[T,220]
    terminal_mask: torch.Tensor       # bool[T]      root is game-over / has no legal action / inactive
    chosen_action_indices: torch.Tensor   # int64[T], -1 for terminal roots


def _capture_graph(graph: torch.cuda.CUDAGraph, pool=None) -> torch.cuda.graph:
    """Capture checked on this thread only: other threads may keep using CUDA meanwhile.  The shard writer's thread
    (``AsyncShardWriter``) waits on its copies of the previous group of games while the next group's engine captures;
    torch's default "global" mode fails that wait with cudaErrorStreamCaptureUnsupported."""
    return torch.cuda.graph(graph, pool=pool, capture_error_mode="thread_local")


class TreeMCTS:
    def __init__(self, net: InferenceNet, num_trees: int, config: TreeMCTSConfig, device=None):
        self.net = net
        self.cfg = config
        self.device = torch.device(device) if device is not None else net.device
        self.num_trees = int(num_trees)
        k = max(1, int(config.leaves_per_wave))
        waves = -(-int(config.num_simulations) // k)
        self.waves = waves
        # with reuse a root starts from the statistics it inherited (up to a few x num_simulations visits)
        # (measured over 300 plies at 4,096 x 200: <= 2.7 M nodes survive a compaction, ~10 M are added per ply)
        hint = config.nodes_per_tree_hint or int(min((waves * k + 2) * 40, 60_000) * (1.5 if config.reuse_subtree else 1))
        self.tree = DeviceTreeBatch(self.num_trees, self.device, exploration_weight=config.exploration_weight,
                                    leaves_per_wave=k, virtual_loss=config.virtual_loss, nodes_per_tree_hint=hint)
        self._advanced = False
        t, slots = self.num_trees, self.num_trees * k
        dev = self.device
        # network batches are whole 64-row tiles (the tcgen05 convolution works on 256-row tile pairs = 64 boards): the
        # buffers are padded, the pad rows hold empty positions whose outputs nobody reads
        tp, sp = -(-t // 64) * 64, -(-slots // 64) * 64
        self._tp, self._sp = tp, sp
        self._root_in = net.new_input(tp)
        self._wave_in = self._root_in if k == 1 else net.new_input(sp)
        self._root_pri = torch.zeros((tp, ACTION_DIM), dtype=torch.float32, device=dev)
        self._root_val = torch.zeros((tp,), dtype=torch.float32, device=dev)
        self._wave_pri = self._root_pri if k == 1 else torch.zeros((sp, ACTION_DIM), dtype=torch.float32, device=dev)
        self._wave_val = self._root_val if k == 1 else torch.zeros((sp,), dtype=torch.float32, device=dev)
        self._wave_graph: Optional[torch.cuda.CUDAGraph] = None
        self._root_graph: Optional[torch.cuda.CUDAGraph] = None
        self.root_graph_launches = self.wave_graph_launches = self.search_extra_launches = 0
        self._first_graph: Optional[torch.cuda.CUDAGraph] = None
        self._last_graph: Optional[torch.cuda.CUDAGraph] = None
        self.evals = 0
        # leaf-batch compaction (set_live / search(live_rows=...)): wave graphs per batch bucket, captured on first use.
        # The row map lives in ONE tensor for the lifetime of the engine and is always attached to the tree (identity =
        # no compaction): the kernels' arguments -- this pointer included -- are frozen into the captured CUDA graphs.
        self._rows = torch.arange(self.num_trees, dtype=torch.int32, device=self.device)
        self._live_set = False
        self.tree.set_tree_rows(self._rows)
        self._bucket_graphs: dict = {}
        self._bucket = self.num_trees
        self._buckets_warm = False

    # ---- leaf-batch compaction: the network only evaluates the live trees' leaves ----------------------------------
    def bucket_for(self, live: int) -> int:
        """Smallest supported wave batch (in trees) that holds `live` trees: 64 / 128 / 256, then multiples of 256 (every
        bucket is a pair of captured CUDA graphs; ``warm_buckets()`` captures the whole ladder once per engine)."""
        t = self.num_trees
        live = max(1, min(int(live), t))
        if live <= 256:
            b = 64
            while b < live:
                b *= 2
        else:
            b = -(-live // 256) * 256
        return t if b >= t else b

    def bucket_ladder(self):
        t = self.num_trees
        return sorted({self.bucket_for(n) for n in [64, 128, 256] + list(range(512, t + 1, 256))} - {t})

    def warm_buckets(self) -> None:
        """Capture the wave graphs of every bucket of the ladder now (between two searches), so that a shrinking batch
        never stops to capture in the middle of an iteration.  One-off cost per engine (~1 s at 4,096 trees); engines are
        kept across iterations (self_play_v1_gpu(engine_cache=...), run_self_play_worker)."""
        if not self.cfg.use_cuda_graph or self._wave_graph is None or self._buckets_warm:
            return
        for b in self.bucket_ladder():
            self._graphs_for(b)
        self._buckets_warm = True

    def set_live(self, active: Optional[torch.Tensor]) -> None:
        """active bool[T] (device) or None.  Live trees get the dense leaf-batch rows 0..n-1 (in tree order), the others
        sit the simulation waves out; no host synchronisation.  Pass an upper bound of n as search(live_rows=...)."""
        if active is None:
            self._rows.copy_(torch.arange(self.num_trees, dtype=torch.int32, device=self.device))
            self._live_set = False
            return
        act = active.to(device=self.device, dtype=torch.bool).view(-1)
        rows = torch.cumsum(act.to(torch.int32), 0, dtype=torch.int32) - 1
        self._rows.copy_(torch.where(act, rows, torch.full_like(rows, -1)))
        self._live_set = True

    # one network evaluation of the pending leaves + expansion (+ backup).  On the tcgen05 paths (net.padded_input) the
    # network input x is the channel-padded bf16 [n,64,6,6] tensor and the select kernel writes it itself (one launch
    # less per wave); other nets (allow_library_convs) take the unpadded input, written by a separate encoding launch.
    def _fused_encode(self, x: torch.Tensor) -> bool:
        return self.net.padded_input

    def _eval_pending(self, root: bool, encoded: bool) -> None:
        tree = self.tree
        x = self._root_in if root else self._wave_in
        pri = self._root_pri if root else self._wave_pri
        val = self._root_val if root else self._wave_val
        if not encoded:
            encode_inputs(tree.pending_states, "bf16_nhwc", out=x)
        self.net.forward_priors(x, tree.pending_states_padded, priors_out=pri, values_out=val)
        tree.complete_pending(pri, val)

    def _root_step(self) -> None:
        fused = self._fused_encode(self._root_in)
        self.tree.prepare_roots(self._root_in if fused else None)
        self._eval_pending(True, fused)

    # A search is: root step, noise, FIRST select, then waves - 1 times [network -> expand+backup -> next select] and
    # one last [network -> expand+backup].  The bracketed parts are one CUDA graph each; expand of wave w and select of
    # wave w + 1 are ONE kernel (lzb_tree_expand_select), so a wave has a single tree kernel.
    def _first_select(self) -> None:
        fused = self._fused_encode(self._wave_in)
        self.tree.select_leaves(self._wave_in if fused else None)
        if not fused:
            encode_inputs(self.tree.pending_states, "bf16_nhwc", out=self._wave_in)

    def _wave_forward(self, bucket: Optional[int]) -> None:
        """The network on the pending leaves: all slots, or only the first bucket * K rows (the live trees' leaves)."""
        tree = self.tree
        n = self._sp if (bucket is None or bucket >= self.num_trees) else int(bucket) * tree.k
        self.net.forward_priors(self._wave_in[:n], tree.pending_states_padded[:n], priors_out=self._wave_pri[:n],
                                values_out=self._wave_val[:n])

    def _wave_mid(self, bucket: Optional[int] = None) -> None:
        tree = self.tree
        fused = self._fused_encode(self._wave_in)
        self._wave_forward(bucket)
        tree.complete_and_select(self._wave_pri, self._wave_val, self._wave_in if fused else None)
        if not fused:
            encode_inputs(tree.pending_states, "bf16_nhwc", out=self._wave_in)

    def _wave_last(self, bucket: Optional[int] = None) -> None:
        self._wave_forward(bucket)
        self.tree.complete_pending(self._wave_pri, self._wave_val)

    def _graphs_for(self, bucket: int):
        """(wave graph, last-wave graph) for a wave batch of `bucket` trees; the full-size pair comes from _capture()."""
        if bucket >= self.num_trees:
            return self._wave_graph, self._last_graph
        pair = self._bucket_graphs.get(bucket)
        if pair is None:
            dev = self.device
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):          # warm-up at this batch size outside the capture; leaves the tree intact:
                self._wave_forward(bucket)         # only the network runs (its outputs are overwritten before use)
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize(dev)
            g_mid, g_last = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
            with _capture_graph(g_mid, pool=self._root_graph.pool()):
                self._wave_mid(bucket)
            with _capture_graph(g_last, pool=self._root_graph.pool()):
                self._wave_last(bucket)
            pair = self._bucket_graphs[bucket] = (g_mid, g_last)
        return pair

    def _capture(self) -> None:
        dev = self.device
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):          # warm up (cuDNN autotune / workspace) outside the capture
            self._root_step()
            self._first_select()
            self._wave_mid()
            self._wave_last()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        from ._lib import launch_count

        # kernels of OURS inside each graph (every replay launches them again; bench.py's gpu_launches)
        c0 = launch_count()
        self._root_graph = torch.cuda.CUDAGraph()
        with _capture_graph(self._root_graph):
            self._root_step()
        c1 = launch_count()
        self._first_graph = torch.cuda.CUDAGraph()
        with _capture_graph(self._first_graph, pool=self._root_graph.pool()):
            self._first_select()
        c2 = launch_count()
        self._wave_graph = torch.cuda.CUDAGraph()
        with _capture_graph(self._wave_graph, pool=self._root_graph.pool()):
            self._wave_mid()
        c3 = launch_count()
        self._last_graph = torch.cuda.CUDAGraph()
        with _capture_graph(self._last_graph, pool=self._root_graph.pool()):
            self._wave_last()
        c4 = launch_count()
        self.root_graph_launches, self.wave_graph_launches = c1 - c0, c3 - c2
        self.search_extra_launches = (c2 - c1) + (c4 - c3) - (c3 - c2)     # per search, on top of waves x wave_graph

    def _apply_root_noise(self) -> None:
        """Dirichlet(alpha) over each root's legal actions mixed with weight epsilon (portable_cpp_mcts.py:180-199,
        v1 root search mcts_gpu.py:1329-1339); Gamma draws come from torch's CUDA generator."""
        cfg = self.cfg
        out = self.tree.root_outputs(with_priors=True)
        legal = out["legal_masks"]
        pri = out["root_priors"]
        alpha = torch.full_like(pri, max(float(cfg.dirichlet_alpha), 1e-8))
        noise = torch._standard_gamma(alpha) * legal.to(torch.float32)
        noise = noise / noise.sum(dim=1, keepdim=True).clamp_min(1e-8)
        eps = min(max(float(cfg.dirichlet_epsilon), 0.0), 1.0)
        mixed = (1.0 - eps) * pri + eps * noise
        many = legal.sum(dim=1, keepdim=True) > 1
        self.tree.set_root_priors(torch.where(many, mixed, pri))

    def advance(self, actions: torch.Tensor, restart_states: Optional[torch.Tensor] = None,
                restart_mask: Optional[torch.Tensor] = None) -> None:
        """After the moves of a ply are chosen: tree t continues from the child reached by ``actions[t]`` (< 0: tree
        kept as it is); slots in ``restart_mask`` start a new game from ``restart_states``.  The next ``search()``
        then skips the reset and every root starts from its inherited subtree.  No-op unless ``reuse_subtree``."""
        if not self.cfg.reuse_subtree:
            return
        self.tree.advance_roots(actions, restart_states, restart_mask)
        self._advanced = True

    @torch.no_grad()
    def search(self, root_states: torch.Tensor, *, active: Optional[torch.Tensor] = None,
               temperatures: Optional[torch.Tensor] = None, add_dirichlet_noise: Optional[bool] = None,
               sample_moves: Optional[bool] = None, live_rows: Optional[int] = None) -> TreeSearchOutput:
        """``live_rows``: after ``set_live(active)``, a host-side UPPER BOUND of the number of live trees -- the simulation
        waves then run the network on ``bucket_for(live_rows)`` rows instead of all trees (same results: the rows of
        trees that sit out were never used)."""
        cfg = self.cfg
        tree = self.tree
        if live_rows is not None and not self._live_set:
            raise RuntimeError("search(live_rows=...) needs set_live(active) first")
        if live_rows is None and self._live_set:
            self.set_live(None)                 # a full-batch search: identity rows
        bucket = self.num_trees if live_rows is None else self.bucket_for(live_rows)
        self._bucket = bucket
        keep = bool(cfg.reuse_subtree) and self._advanced      # roots already in place (advance() after the last move)
        self._advanced = False
        if keep:
            if active is not None:
                tree.set_active(active)
        else:
            tree.reset(root_states, active)
        use_graph = bool(cfg.use_cuda_graph)
        if use_graph and self._wave_graph is None:
            if keep:
                raise RuntimeError("TreeMCTS: the first search must start from reset roots")
            self._capture()
            tree.reset(root_states, active)
        if use_graph:
            self._root_graph.replay()
        else:
            self._root_step()
        if cfg.add_dirichlet_noise if add_dirichlet_noise is None else add_dirichlet_noise:
            self._apply_root_noise()
        if use_graph:
            g_mid, g_last = self._graphs_for(bucket)
            self._first_graph.replay()
            for _ in range(self.waves - 1):
                g_mid.replay()
            g_last.replay()
        else:
            self._first_select()
            for _ in range(self.waves - 1):
                self._wave_mid(bucket)
            self._wave_last(bucket)
        self.evals += self.num_trees + bucket * self.waves * tree.k
        tree.poll_errors()                      # sticky arena / illegal-advance / bad-network flags, without a host sync
        beta = float(cfg.policy_target_prior_pseudocount)
        do_sample = cfg.sample_moves if sample_moves is None else sample_moves
        out = tree.root_outputs(with_priors=(beta > 0.0) or not do_sample)
        visits = out["visit_counts"]
        legal = out["legal_masks"]
        terminal = out["terminal"]
        t = self.num_trees
        if temperatures is None:
            temps = torch.full((t,), float(cfg.temperature), dtype=torch.float32, device=self.device)
        else:
            temps = torch.as_tensor(temperatures, dtype=torch.float32, device=self.device).view(-1)
        selection = policy_from_visits(visits, temps)
        if cfg.policy_target_temperature is None and beta <= 0.0:
            policy = selection
        else:
            t_target = temps if cfg.policy_target_temperature is None else torch.full_like(
                temps, float(cfg.policy_target_temperature))
            policy = policy_from_visits(visits, t_target, legal=legal, priors=out["root_priors"], prior_pseudocount=beta)
        has_mass = selection.sum(dim=1) > 0
        safe = torch.where(has_mass.view(-1, 1), selection, torch.full_like(selection, 1.0 / ACTION_DIM))
        if do_sample:
            chosen = torch.multinomial(safe, num_samples=1).view(-1)
        else:
            chosen = deterministic_action(visits, out["root_action_values"], legal, out["root_priors"])
        chosen = torch.where(has_mass & ~terminal, chosen, torch.full_like(chosen, -1))
        dead = (terminal | ~has_mass).view(-1, 1)
        policy = torch.where(dead, torch.zeros_like(policy), policy)
        return TreeSearchOutput(legal_mask=legal, visit_counts=visits, policy_dense=policy,
                                selection_policy_dense=selection, root_value=out["root_values"],
                                root_action_values=out["root_action_values"], terminal_mask=terminal | ~has_mass,
                                chosen_action_indices=chosen)


def policy_from_visits(visits: torch.Tensor, temperatures: torch.Tensor, legal: Optional[torch.Tensor] = None,
                       priors: Optional[torch.Tensor] = None, prior_pseudocount: float = 0.0) -> torch.Tensor:
    """Batched ``policy_from_visits_and_priors`` (portable_mcts.py:149-204) over rows of the 220-d action space:
    scores = N (+ beta * P, P = root priors clamped at 1e-8 and normalised over the legal actions); policy =
    softmax(log(scores) / T) over scores > 0; one-hot argmax(scores) for T <= 1e-6; rows without mass stay zero."""
    v = visits.to(torch.float32)
    temps = temperatures.view(-1, 1)
    scores = v
    beta = float(prior_pseudocount)
    if beta > 0.0:
        if priors is None or legal is None:
            raise ValueError("prior_pseudocount > 0 needs the root priors and the legal mask")
        lg = legal.to(torch.bool)
        p = torch.where(lg, priors.to(torch.float32).clamp_min(1e-8), torch.zeros_like(v))
        psum = p.sum(dim=1, keepdim=True)
        uniform = lg.to(torch.float32) / lg.sum(dim=1, keepdim=True).clamp_min(1).to(torch.float32)
        p = torch.where(torch.isfinite(psum) & (psum > 0), p / psum.clamp_min(1e-38), uniform)
        scores = v + beta * p
    pos = scores > 0
    logits = torch.where(pos, torch.log(scores.clamp_min(1e-38)) / temps.clamp_min(1e-6), torch.full_like(v, float("-inf")))
    any_pos = pos.any(dim=1, keepdim=True)
    soft = torch.softmax(torch.where(any_pos, logits, torch.zeros_like(logits)), dim=1)
    soft = torch.where(any_pos, soft, torch.zeros_like(soft))
    onehot = torch.zeros_like(v)
    onehot.scatter_(1, scores.argmax(dim=1, keepdim=True), 1.0)
    onehot = torch.where(any_pos, onehot, torch.zeros_like(onehot))
    return torch.where(temps <= 1e-6, onehot, soft)


def deterministic_action(visits: torch.Tensor, action_values: torch.Tensor, legal: torch.Tensor,
                         priors: Optional[torch.Tensor] = None) -> torch.Tensor:
    """max N, then max Q (atol 1e-6), then max P (atol 1e-8), then lowest action index
    (``deterministic_action_from_search``, portable_mcts.py:207-261)."""
    v = torch.where(legal, visits.to(torch.float32), torch.full_like(action_values, -1.0))
    best_n = v.max(dim=1, keepdim=True).values
    cand = v == best_n
    q = torch.where(torch.isfinite(action_values), action_values, torch.full_like(action_values, float("-inf")))
    q = torch.where(cand, q, torch.full_like(q, float("-inf")))
    best_q = q.max(dim=1, keepdim=True).values
    cand = cand & (((q - best_q).abs() <= 1e-6) | (q == best_q))
    if priors is not None:
        p = torch.where(torch.isfinite(priors), priors.to(torch.float32), torch.full_like(q, float("-inf")))
        p = torch.where(cand, p, torch.full_like(p, float("-inf")))
        best_p = p.max(dim=1, keepdim=True).values
        cand = cand & (((p - best_p).abs() <= 1e-8) | (p == best_p))
    return cand.to(torch.int8).argmax(dim=1)
