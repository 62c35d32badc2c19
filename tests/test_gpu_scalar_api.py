"""The object-level half of the v0_core surface (liuzhou_b200/scalar_api.py: GameState / MoveRecord / scalar rule
functions, module.cpp:877-1156) on the GPU kernels, against (1) the legacy-engine golden playouts, (2) the oracle's
scalar engine and (3) -- where oracle/_ref is present -- the reference's own `v0_core` objects, call for call."""
import numpy as np
import pytest

import oracle
from tests._util import STATE_FIELDS, load_golden, load_ref

pytestmark = pytest.mark.gpu


def _legacy_games():
    z = load_golden("legacy_playouts")
    n = z["board"].shape[0]
    mb = np.unpackbits(z["marks_black"], axis=1)[:, :36].reshape(n, 6, 6).astype(bool)
    mw = np.unpackbits(z["marks_white"], axis=1)[:, :36].reshape(n, 6, 6).astype(bool)
    return z, mb, mw


def _state_from_row(v, z, mb, mw, i):
    s = v.GameState()
    s.board = [[int(x) for x in row] for row in z["board"][i]]
    s.marked_black = [(int(r), int(c)) for r, c in zip(*np.nonzero(mb[i]))]
    s.marked_white = [(int(r), int(c)) for r, c in zip(*np.nonzero(mw[i]))]
    sc = z["scalars"][i]
    s.phase, s.current_player = v.Phase(int(sc[0])), v.Player(int(sc[1]))
    (s.pending_marks_required, s.pending_marks_remaining, s.pending_captures_required, s.pending_captures_remaining,
     s.forced_removals_done, s.move_count, s.moves_since_capture) = (int(x) for x in sc[2:9])
    return s


def test_scalar_api_replays_legacy_games():
    """Two full games of the legacy golden set through generate_all_legal_moves_struct / apply_move_struct."""
    from liuzhou_b200 import v0_core as v

    z, mb, mw = _legacy_games()
    gp = z["game_ptr"]
    for g in (0, 7):
        s = v.GameState()
        for i in range(gp[g], gp[g + 1]):
            assert s == _state_from_row(v, z, mb, mw, i), (g, i)
            assert s.is_game_over() == bool(z["over"][i])
            w = s.get_winner()
            assert (0 if w is None else int(w)) == int(z["winner"][i])
            moves = v.generate_all_legal_moves_struct(s)
            want = list(z["legal_idx"][z["legal_ptr"][i]:z["legal_ptr"][i + 1]])
            assert [m.action_index() for m in moves] == want, (g, i)
            a = int(z["chosen"][i])
            if a < 0:
                break
            mv = moves[want.index(a)]
            assert mv.phase == s.phase
            s = v.apply_move_struct(s, mv)


def test_scalar_api_errors_and_per_phase_functions():
    from liuzhou_b200 import v0_core as v

    s = v.GameState()
    assert v.generate_placement_positions(s) == [(r, c) for r in range(6) for c in range(6)]
    assert v.generate_mark_targets(s) == [] and v.generate_movement_moves(s) == []
    with pytest.raises(RuntimeError):            # HasLegalMovementMoves throws outside MOVEMENT (rule_engine.cpp:421-424)
        v.has_legal_movement_moves(s)
    s2 = v.apply_placement_move(s, (2, 3))
    assert s2.board[2][3] == 1 and s2.current_player == v.Player.WHITE and s2.move_count == 0     # counters untouched
    s3 = v.apply_move_struct(s, v.MoveRecord.placement((2, 3)))
    assert s3.move_count == 1 and s3.board == s2.board
    with pytest.raises(RuntimeError):
        v.apply_move_struct(s2, v.MoveRecord.placement((2, 3)))                 # occupied
    with pytest.raises(RuntimeError):
        v.apply_move_struct(s, v.MoveRecord.mark((0, 0)))                       # phase mismatch
    with pytest.raises(RuntimeError):
        v.apply_move_struct(s, v.MoveRecord(v.Phase.PLACEMENT, v.ActionType.MARK, (0, 0)))   # wrong kind for the phase
    moves, codes = v.generate_moves_with_codes(s2)
    assert len(moves) == 35 and codes[0].to_tuple() == (1, 0, 0, 0)
    assert v.encode_action_code(v.MoveRecord.movement((1, 2), (2, 2))).to_tuple() == (2, 8, 14, 0)
    assert v.encode_action_code(v.MoveRecord.process_removal()).to_tuple() == (8, 0, 0, 0)
    assert v.MoveRecord.capture((4, 5)).to_dict() == {"phase": v.Phase.CAPTURE_SELECTION, "action_type": "capture",
                                                      "position": (4, 5)}
    assert v.PLACEMENT == v.Phase.PLACEMENT and v.WHITE == v.Player.WHITE and v.MOVE == v.ActionType.MOVE
    b = v.tensor_batch_from_game_states([s, s2, s3], "cuda:0")
    assert b.board.is_cuda and b.board_size == 6 and bool(b.mask_alive.all())
    back = v.tensor_batch_to_game_states(b)
    assert back[0] == s and back[1] == s2 and back[2] == s3 and back[2].move_count == 1


def _stored_reference_playouts(v):
    """tests/golden/scalar_playouts.npz -- 24 playouts decided by the reference's scalar engine: every state's legal
    action indices and the state each chosen move led to -- through generate_all_legal_moves_struct / apply_move_struct."""
    z = load_golden("scalar_playouts")
    st = {k: z[k] for k in STATE_FIELDS}

    def state(i):
        s = v.GameState()
        s.board = [[int(x) for x in row] for row in st["board"][i]]
        s.marked_black = [(int(r), int(c)) for r, c in zip(*np.nonzero(st["marks_black"][i]))]
        s.marked_white = [(int(r), int(c)) for r, c in zip(*np.nonzero(st["marks_white"][i]))]
        s.phase, s.current_player = v.Phase(int(st["phase"][i])), v.Player(int(st["current_player"][i]))
        for k in STATE_FIELDS[5:]:
            setattr(s, k, int(st[k][i]))
        return s

    gp, checked = z["game_ptr"], 0
    for g in range(len(gp) - 1):
        for i in range(gp[g], gp[g + 1] - 1, 3):
            s, nxt = state(i), state(i + 1)
            moves = v.generate_all_legal_moves_struct(s)
            assert sorted(m.action_index() for m in moves) == list(z["legal_idx"][z["legal_ptr"][i]:z["legal_ptr"][i + 1]])
            got = v.apply_move_struct(s, next(m for m in moves if m.action_index() == int(z["chosen"][i])))
            assert got.board == nxt.board and int(got.phase) == int(nxt.phase)
            assert sorted(got.marked_black) == sorted(nxt.marked_black)
            assert sorted(got.marked_white) == sorted(nxt.marked_white)
            assert int(got.current_player) == int(nxt.current_player)
            for k in STATE_FIELDS[5:]:
                assert getattr(got, k) == getattr(nxt, k), (i, k)
            checked += 1
    assert checked > 500


def test_scalar_api_vs_reference_objects():
    """Call for call against the reference's own v0_core objects on states of oracle playouts (all phases); without
    oracle/_ref, against the playouts the reference's scalar engine stored in tests/golden."""
    from liuzhou_b200 import v0_core as v

    ref = load_ref()
    if ref is None:
        return _stored_reference_playouts(v)
    rv, _ = ref

    def to_ref(s):
        r = rv.GameState()
        r.board = [list(row) for row in s.board]
        r.marked_black, r.marked_white = list(s.marked_black), list(s.marked_white)
        r.phase, r.current_player = rv.Phase(int(s.phase)), rv.Player(int(s.current_player))
        for k in ("forced_removals_done", "move_count", "pending_marks_required", "pending_marks_remaining",
                  "pending_captures_required", "pending_captures_remaining"):
            setattr(r, k, int(getattr(s, k)))
        if hasattr(r, "moves_since_capture"):
            r.moves_since_capture = int(s.moves_since_capture)
        return r

    checked = 0
    for g in range(3):
        trace = oracle.random_playout(123, g, 512, want_trace=True)["trace"]
        s = v.GameState()
        for ply, a in enumerate(trace):
            if ply % 3 == 0:
                r = to_ref(s)
                mine, theirs = v.generate_all_legal_moves_struct(s), rv.generate_all_legal_moves_struct(r)
                def key(m):
                    t = lambda p: None if p is None else (int(p[0]), int(p[1]))      # noqa: E731
                    return (int(m.phase), m.action_type_name, t(m.position), t(m.from_position), t(m.to_position))

                assert [key(m) for m in mine] == [key(t_) for t_ in theirs]
                assert [c.to_tuple() for c in v.encode_action_codes(mine)] == [c.to_tuple() for c in rv.encode_action_codes(theirs)]
                assert v.generate_placement_positions(s) == [tuple(p) for p in rv.generate_placement_positions(r)]
                assert v.generate_mark_targets(s) == [tuple(p) for p in rv.generate_mark_targets(r)]
                assert v.generate_capture_targets(s) == [tuple(p) for p in rv.generate_capture_targets(r)]
                if int(s.phase) == 4:
                    assert v.generate_movement_moves(s) == [(tuple(m[0]), tuple(m[1])) for m in rv.generate_movement_moves(r)]
                checked += 1
            mv = next(m for m in v.generate_all_legal_moves_struct(s) if m.action_index() == int(a))
            nxt = v.apply_move_struct(s, mv)
            if ply % 3 == 0:
                rn = rv.apply_move_struct(to_ref(s), rv.generate_all_legal_moves_struct(to_ref(s))[
                    [m.action_index() for m in v.generate_all_legal_moves_struct(s)].index(int(a))])
                assert nxt.board == [list(row) for row in rn.board]
                assert sorted(nxt.marked_black) == sorted(tuple(p) for p in rn.marked_black)
                assert int(nxt.phase) == int(rn.phase) and int(nxt.current_player) == int(rn.current_player)
                assert nxt.move_count == rn.move_count and nxt.forced_removals_done == rn.forced_removals_done
                assert nxt.pending_marks_remaining == rn.pending_marks_remaining
                assert nxt.pending_captures_remaining == rn.pending_captures_remaining
            s = nxt
    assert checked > 100
