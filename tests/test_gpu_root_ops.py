"""GPU parity of the root-search composite ops (root_pack_sparse_actions, root_finalize_from_visits,
self_play_step_inplace, finalize_trajectory_inplace) vs the oracle and the golden vectors produced by the
reference's CPU `v0_core` (these four are NOT pinned by any reference test -- SURVEY.md section 8c -- so the
golden vectors generated from the reference binary are the pin)."""
import numpy as np
import pytest
import torch

import oracle
from tests._util import STATE_FIELDS, concat_states, golden_states, load_golden, load_ref, to_torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def v0():
    from liuzhou_b200 import v0_core

    return v0_core


def _np(t):
    return t.detach().cpu().numpy()


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def _playout_states(n_games, seed, every=1):
    out = []
    for g in range(n_games):
        trace = oracle.random_playout(seed, g, 512, want_trace=True)["trace"]
        st = oracle.initial_states(1)
        for ply, a in enumerate(trace):
            if ply % every == 0:
                out.append(st)
            st = oracle.apply_move_scalar(st, int(a))
        out.append(st)
    return concat_states(out)


def _check_pack(got, exp):
    assert len(got) == 10
    for i, (g, e) in enumerate(zip(got, exp)):
        g = _np(g)
        assert g.shape == e.shape, (i, g.shape, e.shape)
        if i == 5:
            np.testing.assert_allclose(g, e, rtol=1e-6, atol=1e-7)   # priors: fp32 row-sum order differs
        else:
            assert np.array_equal(g, e), i


def test_root_pack_golden_and_oracle(v0):
    z = load_golden("composites")
    got = v0.root_pack_sparse_actions(_t(z["mask"]), _t(z["probs"]), _t(z["meta"].astype(np.int32)))
    _check_pack(got, [z[f"pack{i}"] for i in range(10)])
    assert got[0].dtype == torch.bool and got[3].dtype == torch.bool and got[4].dtype == torch.int64
    assert got[6].dtype == torch.int32 and got[5].dtype == torch.float32
    # larger random case vs oracle, rows without legal actions included
    st = _playout_states(12, 5)
    mask, meta = oracle.encode_actions_fast(st)
    rng = np.random.default_rng(1)
    mask[rng.random(mask.shape[0]) < 0.1] = False
    probs = (rng.random(mask.shape).astype(np.float32) + 0.01) * mask
    got = v0.root_pack_sparse_actions(_t(mask), _t(probs), _t(meta))
    _check_pack(got, oracle.root_pack_sparse_actions(mask, probs, meta))
    # all rows terminal -> the reference's empty shapes
    got = v0.root_pack_sparse_actions(_t(np.zeros((5, 220), bool)), _t(np.zeros((5, 220), np.float32)),
                                      _t(np.full((5, 220, 4), -1, np.int32)))
    assert got[0].all() and got[1].numel() == 0 and tuple(got[3].shape) == (0, 0) and tuple(got[6].shape) == (0, 0, 4)
    assert tuple(got[8].shape) == (0, 4)


def test_root_finalize_golden_and_oracle(v0):
    z = load_golden("composites")
    b = z["mask"].shape[0]
    got = v0.root_finalize_from_visits(_t(z["pack4"]), _t(z["pack6"]), _t(z["pack3"]), _t(z["visits"]),
                                       _t(z["value_sum"]), _t(z["pack1"]), b, 220, _t(z["temps"]), False)
    np.testing.assert_allclose(_np(got[0]), z["fin0"], rtol=1e-5, atol=1e-7)     # fp32 pow
    for i in (1, 2, 3):
        assert np.array_equal(_np(got[i]), z[f"fin{i}"]), i
    np.testing.assert_allclose(_np(got[4]), z["fin4"], rtol=1e-5, atol=1e-6)
    # low temperature: visits^(1/T) overflows to inf/NaN in the reference too (SURVEY N4); the pick must
    # still follow torch.max semantics (first NaN / first max)
    legal_idx, codes, valid = z["pack4"], z["pack6"], z["pack3"]
    visits = z["visits"].copy()
    temps = np.full((visits.shape[0],), 0.01, np.float32)
    got = v0.root_finalize_from_visits(_t(legal_idx), _t(codes), _t(valid), _t(visits), _t(z["value_sum"]),
                                       _t(z["pack1"]), b, 220, _t(temps), False)
    exp = oracle.root_finalize_from_visits(legal_idx, codes, valid, visits, z["value_sum"], z["pack1"], b, 220, temps)
    assert np.array_equal(_np(got[1]), exp[1])
    assert np.array_equal(_np(got[2]), exp[2])


def test_self_play_step_inplace_golden(v0):
    z = load_golden("composites")
    st = golden_states(z)
    t = to_torch(st, DEV)
    plies, done = _t(z["step_plies_in"]), _t(z["step_done_in"])
    out = v0.self_play_step_inplace(*t, plies, done, _t(z["step_active"]), _t(z["step_codes"]),
                                    _t(z["step_terminal"]), _t(z["step_valid"]), 130, 2.0)
    assert np.array_equal(_np(out[0]), z["step_out0"])
    assert np.array_equal(_np(out[1]), z["step_out1"])
    np.testing.assert_allclose(_np(out[2]), z["step_out2"], rtol=1e-6, atol=1e-7)
    for k, x in zip(STATE_FIELDS, t):
        assert np.array_equal(_np(x).reshape(z[f"step_state_{k}"].shape), z[f"step_state_{k}"]), k
    assert np.array_equal(_np(plies), z["step_plies_out"]) and np.array_equal(_np(done), z["step_done_out"])
    # empty active set
    out = v0.self_play_step_inplace(*t, plies, done, torch.zeros(0, dtype=torch.int64, device=DEV),
                                    torch.zeros((0, 4), dtype=torch.int32, device=DEV),
                                    torch.zeros(0, dtype=torch.bool, device=DEV),
                                    torch.zeros(0, dtype=torch.bool, device=DEV), 130, 2.0)
    assert out[0].numel() == 0 and out[1].numel() == 0


def test_self_play_step_inplace_vs_oracle_large(v0):
    st = _playout_states(40, 21)
    n = st["board"].shape[0]
    rng = np.random.default_rng(2)
    mask, meta = oracle.encode_actions_fast(st)
    plies = st["move_count"].copy()
    done = np.zeros((n,), bool)
    done[::11] = True
    active = np.nonzero(~done)[0].astype(np.int64)
    terminal = ~mask[active].any(1)
    codes = np.full((active.size, 4), -1, np.int32)
    valid = np.zeros((active.size,), bool)
    for j, g in enumerate(active):
        idx = np.nonzero(mask[g])[0]
        if idx.size and rng.random() > 0.03:
            codes[j] = meta[g, rng.choice(idx)]
            valid[j] = True
    t = to_torch(st, DEV)
    t_plies, t_done = _t(plies), _t(done)
    got = v0.self_play_step_inplace(*t, t_plies, t_done, _t(active), _t(codes), _t(terminal), _t(valid), 130, 2.0)
    o_state = {k: np.array(v, copy=True) for k, v in st.items()}
    o_plies, o_done = plies.copy(), done.copy()
    exp = oracle.self_play_step_inplace(o_state, o_plies, o_done, active, codes, terminal, valid, 130, 2.0)
    assert np.array_equal(_np(got[0]), exp[0]) and np.array_equal(_np(got[1]), exp[1])
    np.testing.assert_allclose(_np(got[2]), exp[2], rtol=1e-6, atol=1e-7)
    assert exp[0].size > 30
    for k, x in zip(STATE_FIELDS, t):
        assert np.array_equal(_np(x).reshape(np.asarray(o_state[k]).shape), o_state[k]), k
    assert np.array_equal(_np(t_plies), o_plies) and np.array_equal(_np(t_done), o_done)


def test_finalize_trajectory_inplace_vs_oracle(v0):
    rng = np.random.default_rng(4)
    g_count, t_max = 64, 17
    counts = rng.integers(0, t_max + 1, (g_count,)).astype(np.int64)
    counts[::7] = 0
    sim = np.full((g_count, t_max), -1, np.int64)
    total = int(counts.sum())
    perm = rng.permutation(total)
    k = 0
    for g in range(g_count):
        sim[g, :counts[g]] = perm[k:k + counts[g]]
        k += counts[g]
    signs = rng.choice([-1, 1], total).astype(np.int8)
    slots = rng.permutation(g_count)[:40].astype(np.int64)
    res = rng.choice([-1.0, 0.0, 1.0], slots.size).astype(np.float32)
    soft = rng.random(slots.size).astype(np.float32)
    vt = np.full((total,), np.nan, np.float32)
    svt = np.full((total,), np.nan, np.float32)
    t_vt, t_svt = _t(vt), _t(svt)
    got = v0.finalize_trajectory_inplace(t_vt, t_svt, _t(signs), _t(sim), _t(counts), _t(slots), _t(res), _t(soft))
    exp = oracle.finalize_trajectory_inplace(vt, svt, signs, sim, counts, slots, res, soft)
    for a, e in zip(got, exp):
        assert np.array_equal(_np(a), e)
    assert np.array_equal(_np(t_vt), vt, equal_nan=True) and np.array_equal(_np(t_svt), svt, equal_nan=True)
    # nothing to finalize
    got = v0.finalize_trajectory_inplace(t_vt, t_svt, _t(signs), _t(sim), _t(counts),
                                         torch.zeros(0, dtype=torch.int64, device=DEV),
                                         torch.zeros(0, device=DEV), torch.zeros(0, device=DEV))
    assert got[0].numel() == 0 and _np(got[2]).tolist() == [0, 0, 0]


def test_root_sparse_writeback_vs_oracle_and_reference(v0):
    """a10: `root_sparse_writeback` (module.cpp:365-439) -- the CUDA kernel against the oracle restatement (pinned to the
    reference binary on the CPU) and, where oracle/_ref travelled, against the reference's own op on this GPU."""
    st = _playout_states(8, 31)
    mask, meta = oracle.encode_actions_fast(st)
    rng = np.random.default_rng(9)
    mask[::11] = False
    probs = (rng.random(mask.shape).astype(np.float32) + 0.01) * mask
    (_tm, roots, cnt, valid_mask, legal_idx, priors, code_mat, _f, _c, _p) = oracle.root_pack_sparse_actions(mask, probs, meta)
    policy = rng.random(priors.shape).astype(np.float32) + 0.05
    picks = (rng.integers(0, 1 << 30, roots.size) % cnt).astype(np.int64)
    args = (_t(legal_idx), _t(code_mat), _t(valid_mask), _t(policy), _t(picks), _t(roots), mask.shape[0], 220)
    got = v0.root_sparse_writeback(*args)
    exp = oracle.root_sparse_writeback(legal_idx, code_mat, valid_mask, policy, picks, roots, mask.shape[0], 220)
    assert got[0].dtype == torch.float32 and got[1].dtype == torch.int64 and got[2].dtype == torch.int32
    assert got[3].dtype == torch.bool
    for i, (g, e) in enumerate(zip(got, exp)):
        assert np.array_equal(_np(g), e), i
    ref = load_ref()
    if ref is not None:
        for i, (g, r) in enumerate(zip(got, ref[0].root_sparse_writeback(*args))):
            assert torch.equal(g, r), i
    # no valid roots at all
    empty = v0.root_sparse_writeback(torch.zeros((0, 0), dtype=torch.int64, device=DEV),
                                     torch.zeros((0, 0, 4), dtype=torch.int32, device=DEV),
                                     torch.zeros((0, 0), dtype=torch.bool, device=DEV), torch.zeros((0, 0), device=DEV),
                                     torch.zeros((0,), dtype=torch.int64, device=DEV),
                                     torch.zeros((0,), dtype=torch.int64, device=DEV), 5, 220)
    assert not empty[0].any() and bool((empty[1] == -1).all()) and not empty[3].any()
    with pytest.raises(RuntimeError):
        v0.root_sparse_writeback(*args[:6], -1, 220)


def test_composites_vs_reference_on_gpu(v0):
    """Same ops from the reference's own module executed on CUDA tensors on this box (oracle/_ref); without it, ours
    against the outputs the reference's binaries stored in tests/golden/composites.npz."""
    if load_ref() is None:
        test_root_pack_golden_and_oracle(v0)
        test_root_finalize_golden_and_oracle(v0)
        z = load_golden("composites")
        mi = v0.states_to_model_input(*to_torch(golden_states(z), DEV)[:5])
        assert np.array_equal(np.packbits(_np(mi).astype(np.uint8)), z["model_input"])
        return
    ref_core, _ = load_ref()
    st = _playout_states(10, 77)
    t = to_torch(st, DEV)
    try:
        mask, meta = ref_core.encode_actions_fast(*t[:10], 36, 144, 36, 4)
    except RuntimeError as exc:
        pytest.skip(f"reference CUDA kernels unavailable: {exc}")
    probs = (torch.rand(mask.shape, device=DEV) + 0.01) * mask
    a = v0.root_pack_sparse_actions(mask, probs, meta)
    b = ref_core.root_pack_sparse_actions(mask, probs, meta)
    for i, (x, y) in enumerate(zip(a, b)):
        if i == 5:
            torch.testing.assert_close(x, y, rtol=1e-6, atol=1e-7)
        else:
            assert torch.equal(x, y), i
    visits, value_sum, _ = ref_core.root_puct_allocate_visits(b[5], torch.rand_like(b[5]) * 2 - 1, b[3], 200, 1.0)
    temps = torch.full((b[1].numel(),), 1.0, device=DEV)
    fa = v0.root_finalize_from_visits(b[4], b[6], b[3], visits, value_sum, b[1], mask.size(0), 220, temps, False)
    fb = ref_core.root_finalize_from_visits(b[4], b[6], b[3], visits, value_sum, b[1], mask.size(0), 220, temps, False)
    torch.testing.assert_close(fa[0], fb[0], rtol=1e-5, atol=1e-7)
    assert torch.equal(fa[1], fb[1]) and torch.equal(fa[2], fb[2]) and torch.equal(fa[3], fb[3])
    torch.testing.assert_close(fa[4], fb[4], rtol=1e-5, atol=1e-6)
    mi_a = v0.states_to_model_input(*t[:5])
    mi_b = ref_core.states_to_model_input(*t[:5])
    assert torch.equal(mi_a, mi_b)
