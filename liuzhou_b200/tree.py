"""Device-resident full-tree MCTS (host-side mirror of the reference's ``PortableTreeBatch`` protocol,
/root/reference/v1/cpp/portable_mcts.cpp:437-977 and its Python driver v1/python/portable_cpp_mcts.py:243-390).

All tree state lives in HBM (node arena, structure of arrays); selection / expansion / backup are the
hand-written kernels in csrc/lz_tree.cu.  Shapes are static (``num_trees * leaves_per_wave`` leaf slots per
wave, each with a status), so one simulation wave -- select -> network -> expand+backup -- can be captured
in a CUDA graph.
"""
from __future__ import annotations

import ctypes
from typing import Optional

import torch

from ._lib import check, i64, lib, ptr, require_cuda, stream_ptr

ACTION_DIM = 220
LEAF_EVAL, LEAF_DONE, LEAF_DUPLICATE = 0, 1, 2


class _TreeStruct(ctypes.Structure):
    _fields_ = [(n, ctypes.c_void_p) for n in ("visit", "value_sum", "prior", "info", "first_child", "parent", "state",
                                                "root_value", "counters")] + [("capacity", ctypes.c_int64),
                                                                             ("num_trees", ctypes.c_int64),
                                                                             ("tree_rows", ctypes.c_void_p)]


_ARENA_FIELDS = ("visit", "value_sum", "prior", "info", "first_child", "parent", "state", "root_value", "counters")
FLAG_ARENA, FLAG_ILLEGAL_ADVANCE, FLAG_BAD_NETWORK = 1, 2, 4  # sticky bits of counters[1]


class DeviceTreeBatch:
    """``num_trees`` independent search trees in one node arena on one GPU."""

    def __init__(self, num_trees: int, device="cuda", *, exploration_weight: float = 1.0, leaves_per_wave: int = 1,
                 virtual_loss: float = 1.0, node_capacity: Optional[int] = None,
                 nodes_per_tree_hint: int = 200 * 40) -> None:
        dev = torch.device(device)
        if dev.type != "cuda":
            raise RuntimeError("DeviceTreeBatch needs a CUDA device (no CPU path)")
        if dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        if not (exploration_weight >= 0.0):
            raise RuntimeError("exploration_weight must be finite and non-negative")
        self.device = dev
        self.num_trees = int(num_trees)
        self.k = int(leaves_per_wave)
        self.exploration_weight = float(exploration_weight)
        self.virtual_loss = float(virtual_loss)
        cap = int(node_capacity) if node_capacity is not None else self.num_trees * (1 + int(nodes_per_tree_hint))
        cap = min(cap, 2**31 - 2)
        self.capacity = cap
        t, slots = self.num_trees, self.num_trees * self.k
        with torch.cuda.device(dev):
            self.visit = torch.empty((cap,), dtype=torch.int32, device=dev)
            self.value_sum = torch.empty((cap,), dtype=torch.float64, device=dev)
            self.prior = torch.empty((cap,), dtype=torch.float64, device=dev)
            self.info = torch.empty((cap,), dtype=torch.int32, device=dev)
            self.first_child = torch.empty((cap,), dtype=torch.int32, device=dev)
            self.parent = torch.empty((cap,), dtype=torch.int32, device=dev)
            self.state = torch.empty((cap, 4), dtype=torch.int64, device=dev)
            self.root_value = torch.zeros((t,), dtype=torch.float64, device=dev)
            self.counters = torch.zeros((8,), dtype=torch.int32, device=dev)
            self.leaf_node = torch.full((slots,), -1, dtype=torch.int32, device=dev)
            self.leaf_status = torch.full((slots,), LEAF_DONE, dtype=torch.int32, device=dev)
            # leaf states are allocated in whole 64-row tiles (the tcgen05 network path evaluates multiples of 64 rows;
            # the rows past `slots` stay zero = an empty placement position, evaluated and ignored)
            self.leaf_states_padded = torch.zeros((-(-slots // 64) * 64, 4), dtype=torch.int64, device=dev)
            self.leaf_states = self.leaf_states_padded[:slots]
            # descent paths (LZB_TREE_PATH_STRIDE ints per slot): written by select, consumed by expand + backup
            self.leaf_path = torch.full((slots, 34), -1, dtype=torch.int32, device=dev)
            if self.k == 1:
                self.root_leaf_node, self.root_leaf_status, self.root_leaf_states = (
                    self.leaf_node, self.leaf_status, self.leaf_states)
            else:
                self.root_leaf_node = torch.full((t,), -1, dtype=torch.int32, device=dev)
                self.root_leaf_status = torch.full((t,), LEAF_DONE, dtype=torch.int32, device=dev)
                self.root_leaf_states_padded = torch.zeros((-(-t // 64) * 64, 4), dtype=torch.int64, device=dev)
                self.root_leaf_states = self.root_leaf_states_padded[:t]
            if self.k == 1:
                self.root_leaf_states_padded = self.leaf_states_padded
        self._struct = _TreeStruct()
        for name in _ARENA_FIELDS:
            setattr(self._struct, name, getattr(self, name).data_ptr())
        self._struct.capacity = cap
        self._struct.num_trees = t
        self._pending_is_root = False
        self._tree_rows: Optional[torch.Tensor] = None
        # second arena for advance_roots (subtree reuse); allocated on first use
        self._scratch: Optional[dict] = None
        self._scratch_struct: Optional[_TreeStruct] = None

    # -- protocol ------------------------------------------------------------------------------------
    def reset(self, root_states: torch.Tensor, active: Optional[torch.Tensor] = None) -> None:
        """New search from packed root states int64[T,4] (drops every node of the previous search)."""
        require_cuda(root_states, "root_states")
        if tuple(root_states.shape) != (self.num_trees, 4):
            raise RuntimeError(f"root_states must be int64[{self.num_trees}, 4]")
        rs = root_states.contiguous()
        act = None if active is None else active.to(device=self.device, dtype=torch.bool).contiguous()
        with torch.cuda.device(self.device):
            check(lib().lzb_tree_init_roots(ctypes.byref(self._struct), ptr(rs), ptr(act), stream_ptr(self.device)))

    def _select(self, k: int, roots_only: bool, encode_out: Optional[torch.Tensor]) -> None:
        node, status, states = ((self.root_leaf_node, self.root_leaf_status, self.root_leaf_states) if roots_only
                                else (self.leaf_node, self.leaf_status, self.leaf_states))
        _check_encode_out(encode_out, self.num_trees * k)
        with torch.cuda.device(self.device):
            check(lib().lzb_tree_select(ctypes.byref(self._struct), ctypes.c_int32(k),
                                        ctypes.c_double(self.exploration_weight), ctypes.c_double(self.virtual_loss),
                                        ptr(node), ptr(status), ptr(states), ptr(None if roots_only else self.leaf_path),
                                        ctypes.c_int32(1 if roots_only else 0), ptr(encode_out), stream_ptr(self.device)))

    def prepare_roots(self, encode_out: Optional[torch.Tensor] = None) -> None:
        """Unexpanded, non-terminal, active roots become the pending leaves (one slot per tree, whatever K is);
        roots that kept their subtree through advance_roots() need no evaluation (portable_mcts.cpp:483-513).
        ``encode_out`` (bf16 [T,64,6,6] channels-last): also write the pending roots' network input in the same launch
        (channels 0..15 of the pending rows; channels 16..63 must already be zero, other rows are left untouched)."""
        self._select(1, True, encode_out)
        self._pending_is_root = True

    def _ensure_scratch(self) -> None:
        if self._scratch is not None:
            return
        dev, cap, t = self.device, self.capacity, self.num_trees
        with torch.cuda.device(dev):
            sc = {"visit": torch.empty((cap,), dtype=torch.int32, device=dev),
                  "value_sum": torch.empty((cap,), dtype=torch.float64, device=dev),
                  "prior": torch.empty((cap,), dtype=torch.float64, device=dev),
                  "info": torch.empty((cap,), dtype=torch.int32, device=dev),
                  "first_child": torch.empty((cap,), dtype=torch.int32, device=dev),
                  "parent": torch.empty((cap,), dtype=torch.int32, device=dev),
                  "state": torch.empty((cap, 4), dtype=torch.int64, device=dev),
                  "root_value": torch.zeros((t,), dtype=torch.float64, device=dev),
                  "counters": torch.zeros((8,), dtype=torch.int32, device=dev)}
            self._work = torch.empty((t + cap,), dtype=torch.int32, device=dev)
        st = _TreeStruct()
        for name in _ARENA_FIELDS:
            setattr(st, name, sc[name].data_ptr())
        st.capacity, st.num_trees = cap, t
        self._scratch, self._scratch_struct = sc, st

    def advance_roots(self, actions: torch.Tensor, reset_states: Optional[torch.Tensor] = None,
                      reset_mask: Optional[torch.Tensor] = None) -> None:
        """Subtree reuse after a real move (``PortableTreeBatch.advance_roots``, portable_mcts.cpp:739-768): the child
        reached by ``actions[t]`` (action index; < 0 = keep the tree as it is) becomes the root of tree t with all its
        statistics.  ``reset_mask`` / ``reset_states`` start a new game in the marked slots (fresh unexpanded root).
        The arena is compacted in the same pass, so node indices change and memory use stays bounded over a game.
        No pending evaluation may be outstanding.  Asynchronous; errors surface in ``check_capacity()``."""
        t = self.num_trees
        require_cuda(actions, "actions")
        if actions.numel() != t:
            raise RuntimeError(f"actions must contain one entry per tree ({t})")
        if (reset_states is None) != (reset_mask is None):
            raise RuntimeError("reset_states and reset_mask go together")
        a = actions.to(torch.int32).contiguous()
        rs = rm = None
        if reset_states is not None:
            require_cuda(reset_states, "reset_states")
            if tuple(reset_states.shape) != (t, 4):
                raise RuntimeError(f"reset_states must be int64[{t}, 4]")
            rs = reset_states.contiguous()
            rm = reset_mask.to(device=self.device, dtype=torch.bool).contiguous()
        self._ensure_scratch()
        with torch.cuda.device(self.device):
            check(lib().lzb_tree_advance_roots(ctypes.byref(self._struct), ctypes.byref(self._scratch_struct), ptr(a),
                                               ptr(rs), ptr(rm), ptr(self._work), stream_ptr(self.device)))

    def deactivate(self, tree_indices) -> None:
        """``PortableTreeBatch.deactivate`` (:770-778): the listed trees are skipped by every later call."""
        idx = torch.as_tensor(tree_indices, dtype=torch.int64, device=self.device).view(-1)
        if idx.numel() and (int(idx.min()) < 0 or int(idx.max()) >= self.num_trees):
            raise RuntimeError("deactivate tree index is out of range")
        self.set_active(torch.ones((self.num_trees,), dtype=torch.bool, device=self.device).index_fill_(0, idx, False),
                        only_clear=True)

    def set_active(self, active: torch.Tensor, only_clear: bool = False) -> None:
        """Set (or with ``only_clear`` just clear) the per-tree active flag from bool[T]; no host synchronisation."""
        act = active.to(device=self.device, dtype=torch.bool).view(-1)
        roots = self.info[: self.num_trees]
        bit = 1 << 21                                                     # kInfoInactive (csrc/lz_tree.cu)
        roots.copy_(torch.where(act, roots if only_clear else roots & ~bit, roots | bit))

    def root_states(self) -> torch.Tensor:
        """Packed states int64[T,4] of the current roots (a view into the arena)."""
        return self.state[: self.num_trees]

    def root_status(self) -> dict:
        """``PortableTreeBatch.root_status`` (:780-822) as device tensors."""
        from .engine import _popcount36, packed_status

        p = self.root_states()
        over, winner = packed_status(p)
        meta = (p[:, 0] >> 36) & 0xFFFFFFF
        mask36 = (1 << 36) - 1
        return {"winner": winner.to(torch.int32), "black_pieces": _popcount36(p[:, 0] & mask36).to(torch.int32),
                "white_pieces": _popcount36(p[:, 1] & mask36).to(torch.int32),
                "current_players": (1 - 2 * ((meta >> 3) & 1)).to(torch.int32), "phases": (meta & 7).to(torch.int32),
                "move_counts": ((meta >> 14) & 255).to(torch.int32),
                "moves_since_capture": ((meta >> 22) & 63).to(torch.int32), "game_over": over}

    def select_leaves(self, encode_out: Optional[torch.Tensor] = None) -> None:
        """One descent per leaf slot; ``encode_out`` (bf16 [T*K,64,6,6] channels-last) fuses the input encoding in: channels
        0..15 of the pending rows are written, channels 16..63 must already be zero, other rows are left untouched."""
        self._select(self.k, False, encode_out)
        self._pending_is_root = False

    @property
    def pending_status(self) -> torch.Tensor:
        return self.root_leaf_status if self._pending_is_root else self.leaf_status

    @property
    def pending_states(self) -> torch.Tensor:
        return self.root_leaf_states if self._pending_is_root else self.leaf_states

    @property
    def pending_states_padded(self) -> torch.Tensor:
        """The same rows plus the zero rows up to the next multiple of 64 (network batches are whole 64-row tiles)."""
        return self.root_leaf_states_padded if self._pending_is_root else self.leaf_states_padded

    def complete_pending(self, priors: torch.Tensor, values: torch.Tensor) -> None:
        """priors f32[slots,220] dense over the action space, values f32[slots] (slots = T for roots, T*K for a
        wave); rows of slots whose status is not LEAF_EVAL are ignored.  Roots are expanded without a backup
        (portable_mcts.cpp:575)."""
        root = self._pending_is_root
        k = 1 if root else self.k
        slots = self.num_trees * k
        if priors.dim() != 2 or priors.size(0) < slots or priors.size(1) != ACTION_DIM or values.numel() < slots:
            raise RuntimeError(f"priors must be [>={slots}, 220] and values [>={slots}]")
        require_cuda(priors, "priors")
        p = priors.to(torch.float32).contiguous()
        v = values.to(torch.float32).contiguous()
        node, status = (self.root_leaf_node, self.root_leaf_status) if root else (self.leaf_node, self.leaf_status)
        with torch.cuda.device(self.device):
            check(lib().lzb_tree_expand_backup(ctypes.byref(self._struct), ctypes.c_int32(k), ptr(node), ptr(status),
                                               ptr(p), ptr(v), ctypes.c_int32(0 if root else 1),
                                               ctypes.c_double(self.virtual_loss), ptr(None if root else self.leaf_path),
                                               stream_ptr(self.device)))

    def complete_and_select(self, priors: torch.Tensor, values: torch.Tensor,
                            encode_out: Optional[torch.Tensor] = None) -> None:
        """``complete_pending`` of the current wave followed by ``select_leaves`` of the next one in ONE launch
        (``lzb_tree_expand_select``): trees are independent, so every warp expands, backs up and descends again without a
        grid-wide barrier in between.  Only after ``select_leaves`` (not after ``prepare_roots``).  ``encode_out`` as in
        ``select_leaves``: channels 16..63 must already be zero."""
        if self._pending_is_root:
            raise RuntimeError("complete_and_select follows select_leaves, not prepare_roots")
        slots = self.num_trees * self.k
        if priors.dim() != 2 or priors.size(0) < slots or priors.size(1) != ACTION_DIM or values.numel() < slots:
            raise RuntimeError(f"priors must be [>={slots}, 220] and values [>={slots}]")
        require_cuda(priors, "priors")
        p = priors.to(torch.float32).contiguous()
        v = values.to(torch.float32).contiguous()
        _check_encode_out(encode_out, slots)
        with torch.cuda.device(self.device):
            check(lib().lzb_tree_expand_select(ctypes.byref(self._struct), ctypes.c_int32(self.k), ptr(self.leaf_node),
                                               ptr(self.leaf_status), ptr(p), ptr(v),
                                               ctypes.c_double(self.exploration_weight), ctypes.c_double(self.virtual_loss),
                                               ptr(self.leaf_states), ptr(self.leaf_path), ptr(encode_out),
                                               stream_ptr(self.device)))

    def root_outputs(self, with_priors: bool = True) -> dict:
        t, dev = self.num_trees, self.device
        with torch.cuda.device(dev):
            visits = torch.empty((t, ACTION_DIM), dtype=torch.int32, device=dev)
            q = torch.empty((t, ACTION_DIM), dtype=torch.float32, device=dev)
            rv = torch.empty((t,), dtype=torch.float32, device=dev)
            legal = torch.empty((t, ACTION_DIM), dtype=torch.bool, device=dev)
            term = torch.empty((t,), dtype=torch.bool, device=dev)
            pri = torch.empty((t, ACTION_DIM), dtype=torch.float32, device=dev) if with_priors else None
            check(lib().lzb_tree_root_outputs(ctypes.byref(self._struct), ptr(visits), ptr(q), ptr(rv), ptr(legal),
                                              ptr(term), ptr(pri), stream_ptr(dev)))
        return {"visit_counts": visits, "root_action_values": q, "root_values": rv, "legal_masks": legal,
                "terminal": term, "root_priors": pri}

    def set_root_priors(self, priors: torch.Tensor) -> None:
        if tuple(priors.shape) != (self.num_trees, ACTION_DIM):
            raise RuntimeError("root priors must have shape [trees, 220]")
        p = priors.to(device=self.device, dtype=torch.float32).contiguous()
        with torch.cuda.device(self.device):
            check(lib().lzb_tree_set_root_priors(ctypes.byref(self._struct), ptr(p), stream_ptr(self.device)))

    # -- helpers -------------------------------------------------------------------------------------
    def pending_inputs(self, layout: str = "f32_nchw", out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Model-input planes of every leaf slot (rows of non-pending slots hold stale / zero states)."""
        return encode_inputs(self.pending_states, layout, out)

    def stats(self) -> dict:
        c = self.counters.tolist()
        return {"nodes_used": int(c[0]), "overflow": bool(c[1] & FLAG_ARENA), "flags": int(c[1]),
                "expansions": int(c[2]), "terminal_hits": int(c[3]), "capacity": self.capacity,
                "siblings_scanned": int(c[4]) & 0xFFFFFFFF, "levels_descended": int(c[5]) & 0xFFFFFFFF}

    # -- leaf-batch compaction -----------------------------------------------------------------------
    def set_tree_rows(self, rows: Optional[torch.Tensor]) -> None:
        """rows int32[T] (kept by reference: update it IN PLACE between waves) or None.  In the simulation waves tree t
        uses leaf-batch rows rows[t]*K..; rows[t] < 0 = the tree sits the waves out (finished game).  With the live
        trees' rows dense in [0, n) the network only has to run on ceil64(n) rows (TreeMCTS.search(live_rows=...))."""
        if rows is not None:
            require_cuda(rows, "rows")
            if rows.dtype != torch.int32 or rows.numel() != self.num_trees or not rows.is_contiguous():
                raise RuntimeError(f"tree rows must be a contiguous int32[{self.num_trees}] tensor")
        self._tree_rows = rows
        self._struct.tree_rows = 0 if rows is None else rows.data_ptr()

    # -- error flags ------------------------------------------------------------------------------------
    def _raise_flags(self, flags: int) -> None:
        if flags & FLAG_ILLEGAL_ADVANCE:
            raise RuntimeError("selected action is not a child of the current root")       # the reference's message
        if flags & FLAG_BAD_NETWORK:
            raise RuntimeError("model value is NaN or Inf / model prior is negative, NaN, or Inf")   # portable_mcts.cpp
        if flags & FLAG_ARENA:
            raise RuntimeError(f"tree node arena exhausted (capacity {self.capacity}); raise node_capacity")

    def poll_errors(self) -> None:
        """Non-blocking error check for hot loops: queues an async copy of the sticky flag word into pinned memory and
        raises if an EARLIER copy (whose event has completed) carried a flag -- an error surfaces at most one call late
        and the GPU never waits for the host.  ``check_capacity()`` is the blocking form (end of an iteration)."""
        if getattr(self, "_flag_host", None) is None:
            self._flag_host = torch.zeros((2,), dtype=torch.int32).pin_memory()
            self._flag_event = [None, None]
            self._flag_turn = 0
        i = self._flag_turn
        ev = self._flag_event[i]
        if ev is not None:
            if not ev.query():          # the oldest copy is still in flight: check it next time
                return
            self._raise_flags(int(self._flag_host[i]))
        with torch.cuda.device(self.device):
            self._flag_host[i:i + 1].copy_(self.counters[1:2], non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream(self.device))
        self._flag_event[i] = ev
        self._flag_turn = 1 - i

    def check_capacity(self) -> None:
        self._raise_flags(int(self.counters[1].item()))


def _check_encode_out(encode_out: Optional[torch.Tensor], slots: int) -> None:
    """The fused select kernels write the network input of every pending slot as bf16 channels-last [slots,6,6,64]."""
    if encode_out is not None and (encode_out.dtype != torch.bfloat16 or encode_out.dim() != 4
                                   or encode_out.size(0) < slots or tuple(encode_out.shape[1:]) != (64, 6, 6)
                                   or not encode_out.is_contiguous(memory_format=torch.channels_last)):
        raise RuntimeError(f"encode_out must be bfloat16 [>={slots},64,6,6] in channels_last memory format")


def encode_inputs(packed: torch.Tensor, layout: str = "f32_nchw", out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """packed int64[n,4] -> network input. 'f32_nchw': float32[n,11,6,6]; 'bf16_nhwc': bfloat16[n,11,6,6] in
    channels_last memory format (or, if `out` has 64 channels, the same planes zero-padded to [n,64,6,6])."""
    require_cuda(packed, "packed")
    dev = packed.device
    packed = packed.contiguous()
    n = packed.size(0)
    with torch.cuda.device(dev):
        if layout == "f32_nchw":
            if out is None:
                out = torch.empty((n, 11, 6, 6), dtype=torch.float32, device=dev)
            code = 0
        elif layout == "bf16_nhwc":
            if out is None:
                out = torch.empty((n, 11, 6, 6), dtype=torch.bfloat16, device=dev, memory_format=torch.channels_last)
            if out.size(1) not in (11, 64) or out.dtype != torch.bfloat16:
                raise RuntimeError("bf16_nhwc output must be bfloat16 [n,11,6,6] or channel-padded [n,64,6,6]")
            code = 1 if out.size(1) == 11 else 2          # 2: planes zero-padded to 64 channels (tcgen05 stem conv)
        else:
            raise RuntimeError(f"unknown layout {layout}")
        check(lib().lzb_encode_inputs_packed(ptr(packed), i64(n), ctypes.c_int32(code), ptr(out), stream_ptr(dev)))
    return out


def heads_to_priors(packed: torch.Tensor, log_p1: torch.Tensor, log_p2: torch.Tensor, log_pmc: torch.Tensor,
                    value_logits: torch.Tensor, priors_out: Optional[torch.Tensor] = None,
                    values_out: Optional[torch.Tensor] = None):
    """Fused policy projection (masked softmax over the legal set of each packed state) + bucketed value decode."""
    require_cuda(packed, "packed")
    dev = packed.device
    n = packed.size(0)
    h = [x.reshape(n, 36).to(torch.float32).contiguous() for x in (log_p1, log_p2, log_pmc)]
    vl = value_logits.reshape(n, -1).to(torch.float32).contiguous()
    with torch.cuda.device(dev):
        if priors_out is None:
            priors_out = torch.empty((n, ACTION_DIM), dtype=torch.float32, device=dev)
        if values_out is None:
            values_out = torch.empty((n,), dtype=torch.float32, device=dev)
        check(lib().lzb_heads_to_priors(ptr(packed.contiguous()), i64(n), ptr(h[0]), ptr(h[1]), ptr(h[2]), ptr(vl),
                                        ctypes.c_int32(vl.size(1)), ptr(priors_out), ptr(values_out), stream_ptr(dev)))
    return priors_out, values_out
