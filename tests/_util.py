"""Shared helpers for the test-suite (state samplers that mirror the reference's own tests)."""
from __future__ import annotations

import sys
from pathlib import Path
from types import SimpleNamespace

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
REF_DIR = ROOT / "oracle" / "_ref"
GOLDEN = ROOT / "tests" / "golden"

STATE_FIELDS = (
    "board", "marks_black", "marks_white", "phase", "current_player",
    "pending_marks_required", "pending_marks_remaining",
    "pending_captures_required", "pending_captures_remaining",
    "forced_removals_done", "move_count", "moves_since_capture",
)


def load_ref():
    """Import the reference's own binaries (built by oracle/build_ref.py). Returns (v0_core, portable) or None."""
    if not REF_DIR.is_dir() or not list(REF_DIR.glob("v0_core*.so")):
        return None
    if str(REF_DIR) not in sys.path:
        sys.path.insert(0, str(REF_DIR))
    try:
        import torch  # noqa: F401  (v0_core links libtorch)
        import v0_core
        import _liuzhou_portable_cpp as portable
    except Exception:
        return None
    if not hasattr(v0_core, "encode_actions_fast"):
        return None
    return v0_core, portable


def random_mask_states(n: int, seed: int) -> dict:
    """Same distribution as /root/reference/tests/v0/cuda/test_fast_legal_mask_cuda.py:74-120
    (uniformly random, mostly unreachable boards), generated with numpy instead of torch."""
    rng = np.random.default_rng(seed)
    st = {
        "board": rng.integers(-1, 2, (n, 6, 6)).astype(np.int8),
        "marks_black": rng.integers(0, 2, (n, 6, 6)).astype(np.bool_),
        "marks_white": rng.integers(0, 2, (n, 6, 6)).astype(np.bool_),
        "phase": rng.integers(1, 8, (n,)).astype(np.int64),
        "current_player": (rng.integers(0, 2, (n,)) * -2 + 1).astype(np.int64),
        "pending_marks_required": np.zeros((n,), np.int64),
        "pending_marks_remaining": rng.integers(0, 3, (n,)).astype(np.int64),
        "pending_captures_required": np.zeros((n,), np.int64),
        "pending_captures_remaining": rng.integers(0, 3, (n,)).astype(np.int64),
        "forced_removals_done": rng.integers(0, 3, (n,)).astype(np.int64),
        "move_count": rng.integers(0, 150, (n,)).astype(np.int64),
        "moves_since_capture": rng.integers(0, 40, (n,)).astype(np.int64),
    }
    return st


def sparse_random_states(n: int, seed: int) -> dict:
    """Random boards with varied density and sparse marks: hits the shape / fallback branches that the
    uniform sampler above almost never reaches (full rows, 2x2 blocks, all-in-shape)."""
    rng = np.random.default_rng(seed)
    st = random_mask_states(n, seed + 1)
    dens = rng.random((n, 1, 1))
    u = rng.random((n, 6, 6))
    bias = rng.random((n, 1, 1))
    board = np.where(u < dens * bias, 1, np.where(u < dens, -1, 0)).astype(np.int8)
    # stamp some full lines / squares
    for i in range(0, n, 3):
        v = 1 if rng.random() < 0.5 else -1
        k = rng.integers(0, 3)
        if k == 0:
            board[i, rng.integers(0, 6), :] = v
        elif k == 1:
            board[i, :, rng.integers(0, 6)] = v
        else:
            r, c = rng.integers(0, 5, 2)
            board[i, r:r + 2, c:c + 2] = v
    st["board"] = board
    st["marks_black"] = (rng.random((n, 6, 6)) < 0.08)
    st["marks_white"] = (rng.random((n, 6, 6)) < 0.08)
    return st


def random_apply_batch(n: int, seed: int):
    """Same construction as /root/reference/tests/v0/cuda/test_fast_apply_moves_cuda.py:100-243:
    one synthetic (state, action) pair per row over all 8 action kinds."""
    import random

    rng = random.Random(seed)
    st = {k: [] for k in STATE_FIELDS}
    actions = []
    dirs = [(-1, 0), (1, 0), (0, -1), (0, 1)]
    for _ in range(n):
        board = np.array([rng.choice([-1, 0, 1]) for _ in range(36)], np.int8)
        mb = np.zeros(36, np.bool_)
        mw = np.zeros(36, np.bool_)
        cur = rng.choice([-1, 1])
        phase = 1
        pm_req = pm_rem = pc_req = pc_rem = forced = 0
        kind = rng.choice([1, 2, 3, 4, 5, 6, 7, 8])
        cell = rng.randrange(36)
        if kind == 1:
            phase = 1
            board[cell] = 0
            action = (kind, cell, 0, 0)
        elif kind == 3:
            phase = 2
            board[cell] = -cur
            pm_req = pm_rem = rng.choice([1, 2])
            action = (kind, cell, 0, 0)
        elif kind == 8:
            phase = 3
            board[0] = 1
            board[1] = -1
            mb[0] = True
            mw[1] = True
            action = (kind, 0, 0, 0)
        elif kind == 5:
            phase = 6
            cur = -1
            board[0] = 1
            action = (kind, 0, 0, 0)
        elif kind == 2:
            phase = 4
            while True:
                origin = rng.randrange(36)
                d = rng.randrange(4)
                r, c = divmod(origin, 6)
                rt, ct = r + dirs[d][0], c + dirs[d][1]
                if 0 <= rt < 6 and 0 <= ct < 6:
                    break
            board[:] = 0
            board[origin] = cur
            action = (kind, origin, d, 0)
        elif kind == 7:
            phase = 4
            board[cell] = -cur
            action = (kind, cell, 0, 0)
        elif kind == 4:
            phase = 5
            board[cell] = -cur
            if -cur == -1:
                mw[cell] = True
            else:
                mb[cell] = True
            pc_req = pc_rem = rng.choice([1, 2])
            action = (kind, cell, 0, 0)
        else:  # 6
            phase = 7
            board[cell] = -cur
            action = (kind, cell, 0, 0)
        vals = dict(board=board.reshape(6, 6), marks_black=mb.reshape(6, 6), marks_white=mw.reshape(6, 6),
                    phase=phase, current_player=cur, pending_marks_required=pm_req, pending_marks_remaining=pm_rem,
                    pending_captures_required=pc_req, pending_captures_remaining=pc_rem,
                    forced_removals_done=forced, move_count=rng.randrange(0, 100),
                    moves_since_capture=rng.randrange(0, 30))
        for k in STATE_FIELDS:
            st[k].append(vals[k])
        actions.append(action)
    out = {}
    for k in STATE_FIELDS:
        arr = np.stack(st[k]) if k in ("board", "marks_black", "marks_white") else np.array(st[k], np.int64)
        out[k] = arr
    return out, np.array(actions, np.int32), np.arange(n, dtype=np.int64)


def state_obj(st: dict, i: int = 0):
    """Python object with the attributes the reference's `StateFromPython` reads (portable_mcts.cpp:62-141)."""
    return SimpleNamespace(
        board=[[int(v) for v in row] for row in np.asarray(st["board"][i]).reshape(6, 6)],
        phase=int(st["phase"][i]),
        current_player=int(st["current_player"][i]),
        marked_black=[(int(r), int(c)) for r, c in zip(*np.nonzero(np.asarray(st["marks_black"][i]).reshape(6, 6)))],
        marked_white=[(int(r), int(c)) for r, c in zip(*np.nonzero(np.asarray(st["marks_white"][i]).reshape(6, 6)))],
        forced_removals_done=int(st["forced_removals_done"][i]),
        move_count=int(st["move_count"][i]),
        pending_marks_required=int(st["pending_marks_required"][i]),
        pending_marks_remaining=int(st["pending_marks_remaining"][i]),
        pending_captures_required=int(st["pending_captures_required"][i]),
        pending_captures_remaining=int(st["pending_captures_remaining"][i]),
        moves_since_capture=int(st["moves_since_capture"][i]),
    )


def dict_to_state(d: dict) -> dict:
    """Inverse of state_obj for the dicts returned by the reference's `StateToPython` (portable_mcts.cpp:143-166)."""
    mb = np.zeros((1, 6, 6), np.bool_)
    mw = np.zeros((1, 6, 6), np.bool_)
    for r, c in d["marked_black"]:
        mb[0, r, c] = True
    for r, c in d["marked_white"]:
        mw[0, r, c] = True
    st = {"board": np.array(d["board"], np.int8).reshape(1, 6, 6), "marks_black": mb, "marks_white": mw}
    for k in STATE_FIELDS[3:]:
        st[k] = np.array([int(d[k])], np.int64)
    return st


def concat_states(states: list) -> dict:
    return {k: np.concatenate([s[k] for s in states], 0) for k in STATE_FIELDS}


def states_equal(a: dict, b: dict) -> bool:
    return all(np.array_equal(np.asarray(a[k]).reshape(np.asarray(b[k]).shape), np.asarray(b[k])) for k in STATE_FIELDS)


def to_torch(st: dict, device="cpu"):
    import torch

    return [torch.from_numpy(np.ascontiguousarray(st[k])).to(device) for k in STATE_FIELDS]


def fake_net(model_inputs, legal_masks, salt):
    """Deterministic stand-in for the network used by the tree-MCTS parity tests and golden vectors:
    priors / value are a pure function of the model-input planes (so every implementation that reaches the
    same leaf gets the same 'network output')."""
    n = model_inputs.shape[0]
    pri = np.zeros((n, 220), np.float32)
    val = np.zeros((n,), np.float32)
    for i in range(n):
        b = np.packbits(model_inputs[i].astype(np.uint8).ravel())
        h = (int.from_bytes(b.tobytes()[:8], "little") ^ (int(b.sum()) * 2654435761) ^ salt) & 0xFFFFFFFF
        rng = np.random.default_rng(h)
        p = (rng.random(220).astype(np.float32) + 0.05) * (legal_masks[i] != 0)
        s = p.sum()
        pri[i] = p / s if s > 0 else p
        val[i] = np.float32(rng.random() * 2 - 1)
    return pri, val


def bf16_ulp(x):
    """One bf16 step (8 significant bits) at |x|, in fp64; 0 at 0.  x: a torch tensor."""
    import torch

    a = x.double().abs()
    e = torch.floor(torch.log2(torch.where(a > 0, a, torch.ones_like(a))))
    return torch.where(a > 0, torch.exp2(e - 7), torch.zeros_like(a))


def load_golden(name: str) -> dict:
    with np.load(GOLDEN / f"{name}.npz") as z:
        return {k: z[k] for k in z.files}


def golden_states(z: dict, prefix: str = "") -> dict:
    return {k: z[f"{prefix}{k}"] for k in STATE_FIELDS}
