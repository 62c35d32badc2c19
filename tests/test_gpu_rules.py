"""GPU parity (through the C ABI) of the rule-engine kernels vs the oracle, the committed golden vectors and --
when oracle/_ref travelled to the box -- the reference's own CUDA kernels running on the same B200.

Bar: bit-exact (torch.equal) for every integer / byte / index output.
"""
import numpy as np
import pytest
import torch

import oracle
from tests._util import (STATE_FIELDS, concat_states, golden_states, load_golden, load_ref, random_apply_batch,
                         random_mask_states, sparse_random_states, to_torch)

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def v0():
    from liuzhou_b200 import v0_core

    return v0_core


@pytest.fixture(scope="module")
def native():
    from liuzhou_b200 import native

    return native


def _np(t):
    return t.detach().cpu().numpy()


def _cmp_states(got_tensors, expect: dict):
    for k, t in zip(STATE_FIELDS, got_tensors):
        e = np.asarray(expect[k])
        assert np.array_equal(_np(t).reshape(e.shape), e), k


@pytest.mark.parametrize("sampler,seed", [(random_mask_states, 0xF00DCAFE), (sparse_random_states, 0x5EED)])
@pytest.mark.parametrize("aux", [1, 4])
def test_encode_actions_fast_vs_oracle(v0, sampler, seed, aux):
    st = sampler(10_000, seed)
    mask, meta = v0.encode_actions_fast(*to_torch(st, DEV)[:10], 36, 144, 36, aux)
    o_mask, o_meta = oracle.encode_actions_fast(st, 36, 144, 36, aux)
    assert mask.dtype == torch.bool and meta.dtype == torch.int32
    assert np.array_equal(_np(mask), o_mask)
    assert np.array_equal(_np(meta), o_meta)


def test_encode_actions_fast_golden(v0):
    z = load_golden("encode_actions")
    st = golden_states(z)
    for aux in (1, 4):
        mask, meta = v0.encode_actions_fast(*to_torch(st, DEV)[:10], 36, 144, 36, aux)
        total = 216 + aux
        assert np.array_equal(_np(mask), np.unpackbits(z[f"mask_aux{aux}"], axis=1)[:, :total].astype(bool))
        assert np.array_equal(_np(meta), z[f"meta_aux{aux}"].astype(np.int32))


def test_encode_actions_edge_cases(v0):
    # empty batch
    st = oracle.empty_states(0)
    mask, meta = v0.encode_actions_fast(*to_torch(st, DEV)[:10], 36, 144, 36, 4)
    assert tuple(mask.shape) == (0, 220) and tuple(meta.shape) == (0, 220, 4)
    # non-contiguous views are accepted (reference calls .contiguous())
    st = random_mask_states(64, 1)
    t = to_torch(st, DEV)
    t2 = [x.repeat_interleave(2, 0)[::2] for x in t]
    m1, _ = v0.encode_actions_fast(*t[:10], 36, 144, 36, 4)
    m2, _ = v0.encode_actions_fast(*t2[:10], 36, 144, 36, 4)
    assert torch.equal(m1, m2)
    # CPU tensors are refused loudly (no CPU fallback)
    with pytest.raises(RuntimeError):
        v0.encode_actions_fast(*to_torch(st, "cpu")[:10], 36, 144, 36, 4)


def _playout_states(n_games, seed):
    out = []
    for g in range(n_games):
        trace = oracle.random_playout(seed, g, 512, want_trace=True)["trace"]
        st = oracle.initial_states(1)
        for a in trace:
            out.append(st)
            st = oracle.apply_move_scalar(st, int(a))
        out.append(st)
    return concat_states(out)


def test_batch_apply_moves_vs_oracle(v0):
    # (1) reference sampler (legal + silently ignored illegal rows), (2) all legal children of reachable
    # states, (3) garbage states x garbage codes incl. out-of-range parents
    st1, codes1, par1 = random_apply_batch(10_000, 0xA11CEB0B)
    ps = _playout_states(30, 8)
    m, meta = oracle.encode_actions_fast(ps)
    rows, cols = np.nonzero(m)
    st3 = sparse_random_states(8000, 4)
    rng = np.random.default_rng(3)
    codes3 = np.stack([rng.integers(0, 10, 8000), rng.integers(-2, 38, 8000), rng.integers(-1, 5, 8000),
                       rng.integers(-1, 36, 8000)], 1).astype(np.int32)
    par3 = rng.integers(0, 8000, 8000).astype(np.int64)
    for st, codes, parents in ((st1, codes1, par1), (ps, meta[rows, cols], rows.astype(np.int64)), (st3, codes3, par3)):
        out = v0.batch_apply_moves(*to_torch(st, DEV), torch.from_numpy(codes).to(DEV), torch.from_numpy(parents).to(DEV))
        assert len(out) == 12 and out[0].dtype == torch.int8 and out[1].dtype == torch.bool and out[3].dtype == torch.int64
        _cmp_states(out, oracle.batch_apply_moves(st, codes, parents))


def test_batch_apply_moves_thread_kernel_large_batches(v0):
    """N >= 8,192 runs the thread-per-action kernel (word loads / stores), smaller N the warp-per-action one: both must
    give the oracle's children on garbage states x garbage codes (bytes outside -1/0/1 carried over, illegal actions and
    out-of-range parents ignored), on every legal child of reachable states, in place, and on a 2-byte-misaligned view
    (which has to fall back to the byte kernel)."""
    rng = np.random.default_rng(12)
    st = sparse_random_states(6000, 9)
    st["board"] = st["board"].copy()
    st["board"].reshape(-1)[rng.integers(0, st["board"].size, 3000)] = rng.integers(-5, 6, 3000).astype(np.int8)   # garbage bytes
    n = 40_000
    codes = np.stack([rng.integers(0, 10, n), rng.integers(-2, 38, n), rng.integers(-1, 5, n), rng.integers(-1, 36, n)],
                     1).astype(np.int32)
    parents = rng.integers(-2, 6003, n).astype(np.int64)                    # a few out of range
    t = to_torch(st, DEV)
    big = v0.batch_apply_moves(*t, torch.from_numpy(codes).to(DEV), torch.from_numpy(parents).to(DEV))
    small = v0.batch_apply_moves(*t, torch.from_numpy(codes[:4000]).to(DEV), torch.from_numpy(parents[:4000]).to(DEV))
    ok = (parents >= 0) & (parents < 6000)
    want = oracle.batch_apply_moves(st, codes, np.where(ok, parents, 0))
    for k, b_, s_ in zip(STATE_FIELDS, big, small):
        e = np.asarray(want[k]).reshape(_np(b_).shape)
        assert np.array_equal(_np(b_)[ok], e[ok]), k                         # rows of skipped parents are unspecified
        assert np.array_equal(_np(s_)[ok[:4000]], e[:4000][ok[:4000]]), k
    # all legal children of reachable states (> 8,192 rows)
    ps = _playout_states(12, 33)
    m, meta = oracle.encode_actions_fast(ps)
    rows, cols = np.nonzero(m)
    assert rows.size > 8192
    out = v0.batch_apply_moves(*to_torch(ps, DEV), torch.from_numpy(meta[rows, cols]).to(DEV),
                               torch.from_numpy(rows.astype(np.int64)).to(DEV))
    _cmp_states(out, oracle.batch_apply_moves(ps, meta[rows, cols], rows.astype(np.int64)))
    # in place, one legal action per slot, > 8,192 slots
    big_ps = concat_states([ps] * 8)
    nb = big_ps["board"].shape[0]
    mb_, metab = oracle.encode_actions_fast(big_ps)
    has = mb_.any(1)
    slots = np.nonzero(has)[0].astype(np.int64)
    assert slots.size > 8192
    pick = np.array([np.nonzero(mb_[i])[0][(7 * i) % mb_[i].sum()] for i in slots])
    codes_i = metab[slots, pick]
    ti = to_torch(big_ps, DEV)
    v0.batch_apply_moves_inplace(*ti, torch.from_numpy(codes_i).to(DEV), torch.from_numpy(slots).to(DEV))
    _cmp_states(ti, oracle.batch_apply_moves_inplace(big_ps, codes_i, slots))
    # a byte-misaligned board view -> byte kernel, same result
    raw = torch.zeros((nb * 36 + 2,), dtype=torch.int8, device=DEV)
    view = raw[2:].view(nb, 6, 6)
    tv = to_torch(big_ps, DEV)
    view.copy_(tv[0])
    tv[0] = view
    out_v = v0.batch_apply_moves(*tv, torch.from_numpy(codes_i).to(DEV), torch.from_numpy(slots).to(DEV))
    _cmp_states(out_v, oracle.batch_apply_moves(big_ps, codes_i, slots))


def test_batch_apply_moves_golden(v0):
    z = load_golden("apply_moves")
    out = v0.batch_apply_moves(*to_torch(golden_states(z, "in_"), DEV), torch.from_numpy(z["codes"]).to(DEV),
                               torch.from_numpy(z["parents"]).to(DEV))
    _cmp_states(out, {k: z[f"out_{k}"] for k in STATE_FIELDS})


def test_batch_apply_moves_inplace(v0):
    ps = _playout_states(20, 21)
    n = ps["board"].shape[0]
    m, meta = oracle.encode_actions_fast(ps)
    rng = np.random.default_rng(0)
    slots, codes = [], []
    for i in range(n):
        idx = np.nonzero(m[i])[0]
        if idx.size and rng.random() < 0.7:
            slots.append(i)
            codes.append(meta[i, rng.choice(idx)])
    slots = np.array(slots, np.int64)
    codes = np.array(codes, np.int32)
    t = to_torch(ps, DEV)
    v0.batch_apply_moves_inplace(*t, torch.from_numpy(codes).to(DEV), torch.from_numpy(slots).to(DEV))
    _cmp_states(t, oracle.batch_apply_moves_inplace(ps, codes, slots))
    # empty action list is a no-op
    v0.batch_apply_moves_inplace(*t, torch.zeros((0, 4), dtype=torch.int32, device=DEV),
                                 torch.zeros((0,), dtype=torch.int64, device=DEV))


def test_states_to_model_input(v0):
    st = concat_states([random_mask_states(3000, 11), _playout_states(5, 2)])
    got = v0.states_to_model_input(*to_torch(st, DEV)[:5])
    assert got.dtype == torch.float32 and tuple(got.shape[1:]) == (11, 6, 6)
    assert np.array_equal(_np(got), oracle.states_to_model_input(st))


def test_project_policy_logits_fast(v0):
    rng = np.random.default_rng(9)
    st = _playout_states(6, 9)
    mask, _ = oracle.encode_actions_fast(st)
    n = mask.shape[0]
    mask[::13] = False
    heads = [torch.log_softmax(torch.from_numpy(rng.standard_normal((n, 36)).astype(np.float32)), 1) for _ in range(3)]
    p, l = v0.project_policy_logits_fast(*(h.to(DEV) for h in heads), torch.from_numpy(mask).to(DEV), 36, 144, 36, 4)
    op, ol = oracle.project_policy_logits_fast(*(h.numpy() for h in heads), mask)
    # floating point: fp32 softmax, tolerance 1e-5 relative (north_star)
    np.testing.assert_allclose(_np(p), op, rtol=1e-5, atol=1e-7)
    fin = np.isfinite(ol)
    assert np.array_equal(np.isfinite(_np(l)), fin)
    np.testing.assert_allclose(_np(l)[fin], ol[fin], rtol=1e-6, atol=1e-6)
    z = load_golden("composites")
    p, _ = v0.project_policy_logits_fast(*(torch.from_numpy(z[f"head{i}"]).to(DEV) for i in range(3)),
                                         torch.from_numpy(z["mask"]).to(DEV), 36, 144, 36, 4)
    np.testing.assert_allclose(_np(p), z["proj_probs"], rtol=1e-5, atol=1e-7)


@pytest.mark.parametrize("r,m,sims,c", [(64, 40, 200, 1.0), (16, 7, 64, 1.5), (8, 220, 800, 1.0), (4, 1, 16, 1.0),
                                         (512, 33, 128, 1.0), (3, 300, 50, 2.0), (0, 5, 10, 1.0)])
def test_root_puct_vs_oracle(v0, r, m, sims, c):
    rng = np.random.default_rng(5 + r + m)
    valid = rng.random((r, m)) < 0.8
    if r:
        valid[:, 0] = True
        valid[-1, :] = False  # a root without any valid action: stays all-zero like the reference
    pri = rng.random((r, m)).astype(np.float32) * valid
    pri = (pri / np.maximum(pri.sum(1, keepdims=True), 1e-8)).astype(np.float32)
    leaf = ((rng.random((r, m)).astype(np.float32) * 2 - 1) * valid).astype(np.float32)
    leaf[: r // 2] = np.round(leaf[: r // 2] * 4) / 4          # exact ties -> lowest-index tie-break
    if r >= 4:
        pri[: r // 4] = (valid[: r // 4] / np.maximum(valid[: r // 4].sum(1, keepdims=True), 1)).astype(np.float32)
    v, w, rv = v0.root_puct_allocate_visits(torch.from_numpy(pri).to(DEV), torch.from_numpy(leaf).to(DEV),
                                            torch.from_numpy(valid).to(DEV), sims, c)
    ov, ow, orv = oracle.root_puct_allocate_visits(pri, leaf, valid, sims, c)
    assert np.array_equal(_np(v), ov)            # identical visit counts
    assert np.array_equal(_np(w), ow)            # identical fp32 accumulation order
    np.testing.assert_allclose(_np(rv), orv, rtol=1e-5, atol=1e-6)
    if r:
        assert _np(v).sum(1)[:-1].tolist() == [float(sims)] * (r - 1)


def test_root_puct_golden(v0):
    z = load_golden("root_puct")
    for tag in "abc":
        v, w, rv = v0.root_puct_allocate_visits(
            torch.from_numpy(z[f"{tag}_priors"]).to(DEV), torch.from_numpy(z[f"{tag}_leaf"]).to(DEV),
            torch.from_numpy(z[f"{tag}_valid"]).to(DEV), int(z[f"{tag}_sims"]), float(z[f"{tag}_c"]))
        assert np.array_equal(_np(v), z[f"{tag}_visits"])
        assert np.array_equal(_np(w), z[f"{tag}_value_sum"])
        np.testing.assert_allclose(_np(rv), z[f"{tag}_root_values"], rtol=1e-5, atol=1e-6)


def test_pack_unpack_and_native_rules(native):
    st = _playout_states(30, 33)
    n = st["board"].shape[0]
    packed = native.pack_states(to_torch(st, DEV))
    assert tuple(packed.shape) == (n, 4)
    _cmp_states(native.unpack_states(packed), st)          # lossless round trip on reachable states
    for scalar in (True, False):
        words, counts = native.legal_masks(packed, scalar_semantics=scalar)
        mask = _np(native.mask_words_to_bool(words))
        if scalar:
            for i in range(0, n, 5):
                assert list(np.nonzero(mask[i])[0]) == oracle.legal_actions(st, i)[0]
        else:
            assert np.array_equal(mask, oracle.encode_actions_fast(st)[0])
        assert np.array_equal(_np(counts), mask.sum(1))
    # apply every legal action of the non-terminal states
    mask = oracle.encode_actions_fast(st)[0]
    rows, cols = np.nonzero(mask)
    keep = np.array([not oracle.is_game_over(st, int(r)) for r in rows])
    rows, cols = rows[keep], cols[keep]
    children = native.apply_actions(packed, torch.from_numpy(cols.astype(np.int32)).to(DEV),
                                    torch.from_numpy(rows.astype(np.int64)).to(DEV))
    got = native.unpack_states(children)
    meta = oracle.encode_actions_fast(st)[1]
    _cmp_states(got, oracle.batch_apply_moves(st, meta[rows, cols], rows.astype(np.int64)))
    init = native.unpack_states(native.init_states(7, DEV))
    _cmp_states(init, oracle.initial_states(7))


def test_playout_small_vs_oracle(native):
    """Config 2 at a size the oracle finishes in seconds: every game's length, outcome, final state and the
    chained hash of ALL intermediate states are identical."""
    n = 2048
    pb = native.PlayoutBatch(n, seed=20260314, device=DEV, track_hash=True)
    pb.run(max_steps=40)          # resume across launches
    pb.run(max_steps=1)
    pb.run()
    assert int((pb.result == 2).sum()) == 0
    plies, res, hashes = _np(pb.plies), _np(pb.result), _np(pb.hash).view(np.uint64)
    final = native.unpack_states(pb.packed)
    final = {k: _np(t) for k, t in zip(STATE_FIELDS, final)}
    for g in range(n):
        exp = oracle.random_playout(20260314, g, 512)
        assert plies[g] == exp["plies"] and res[g] == exp["result"], g
        assert int(hashes[g]) == exp["hash"], g
        if g % 64 == 0:
            for k in STATE_FIELDS:
                assert np.array_equal(final[k][g], np.asarray(exp["final"][k])[0]), (g, k)


def test_playout_full_size_properties(native):
    """BASELINE config 2 at full size (65,536 games): size-independent properties -- all games finish,
    lengths / outcome mix match the engine's known statistics, a re-run is bit-identical (determinism), a
    different launch chunking gives the identical result, and EVERY one of the 65,536 games matches the oracle's
    replay of the same seeded game: length, outcome and the hash chained over every state of the game."""
    n = 65_536
    pb = native.PlayoutBatch(n, seed=20260314, device=DEV, track_hash=True)
    pb.run()
    assert int((pb.result == 2).sum()) == 0
    plies = pb.plies.to(torch.float64)
    assert 120.0 < float(plies.mean()) < 135.0
    assert int(pb.plies.max()) <= 144 + 1
    draws = float((pb.result == 0).to(torch.float64).mean())
    assert draws > 0.85
    h1, p1, r1 = pb.hash.clone(), pb.plies.clone(), pb.result.clone()
    pb.reset()
    for _ in range(200):
        pb.run(max_steps=1)
    assert torch.equal(pb.hash, h1) and torch.equal(pb.plies, p1) and torch.equal(pb.result, r1)
    o_plies, o_res, o_hash = oracle.random_playouts_each(20260314, 0, n)
    assert np.array_equal(_np(p1).astype(np.int32), o_plies)
    assert np.array_equal(_np(r1).astype(np.int8), o_res)
    assert np.array_equal(_np(h1).view(np.uint64), o_hash)


def test_vs_reference_cuda_kernels(v0):
    """Where oracle/_ref holds the reference's own CUDA build: run ITS kernels on this B200 on the reference tests'
    samplers (10,000 states / 10,000 actions) and require torch.equal with ours.  Without it: ours against the outputs
    the reference's binaries stored in tests/golden (encode_actions, apply_moves, root_puct)."""
    if load_ref() is None:
        test_encode_actions_fast_golden(v0)
        test_batch_apply_moves_golden(v0)
        test_root_puct_golden(v0)
        return
    ref_core, _ = load_ref()
    st = random_mask_states(10_000, 0xF00DCAFE)
    t = to_torch(st, DEV)
    try:
        r_mask, r_meta = ref_core.encode_actions_fast(*t[:10], 36, 144, 36, 1)
    except RuntimeError as exc:  # reference built without CUDA kernels
        pytest.skip(f"reference CUDA kernels unavailable: {exc}")
    mask, meta = v0.encode_actions_fast(*t[:10], 36, 144, 36, 1)
    assert torch.equal(mask, r_mask) and torch.equal(meta, r_meta)
    st, codes, parents = random_apply_batch(10_000, 0xA11CEB0B)
    t = to_torch(st, DEV)
    c, p = torch.from_numpy(codes).to(DEV), torch.from_numpy(parents).to(DEV)
    for a, b in zip(v0.batch_apply_moves(*t, c, p), ref_core.batch_apply_moves(*t, c, p)):
        assert torch.equal(a, b.to(a.dtype))
    rng = np.random.default_rng(1)
    valid = torch.from_numpy(rng.random((256, 48)) < 0.8).to(DEV)
    valid[:, 0] = True
    pri = torch.rand((256, 48), device=DEV) * valid
    pri = pri / pri.sum(1, keepdim=True)
    leaf = (torch.rand((256, 48), device=DEV) * 2 - 1) * valid
    leaf[:128] = torch.round(leaf[:128] * 4) / 4
    for sims in (200, 800):
        a = v0.root_puct_allocate_visits(pri, leaf, valid, sims, 1.0)
        b = ref_core.root_puct_allocate_visits(pri, leaf, valid, sims, 1.0)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
        torch.testing.assert_close(a[2], b[2], rtol=1e-5, atol=1e-6)
