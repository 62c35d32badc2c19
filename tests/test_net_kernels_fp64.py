"""The network's floating-point kernels against plain fp64 references of the same operations.

heads_tail_kernel (csrc/lz_nn.cu) and bn_relu_kernel are compared element by element with an fp64 evaluation of what
they compute.  Every tolerance is an error bound derived from the data: the reference also evaluates, in fp64, a
magnitude term (the same expression on |weights| and |inputs|), and a test asserts |kernel - ref| <= c * u * magnitude,
with u the unit roundoff of the step (U_TF32 for a TF32 operand, K * U_FP32 for fp32 accumulation over K terms) and a
stated c <= 4.  The CPU tests pin the reference itself (to the PyTorch modules in fp64, to the oracle's projection) and
the host-side weight packers to their documented layouts.
"""
import copy
import ctypes
import math

import numpy as np
import pytest
import torch

import oracle
from tests._util import bf16_ulp, concat_states, to_torch

DEV = "cuda:0"
U_TF32 = 2.0 ** -11          # cvt.rna.tf32.f32: 10 stored mantissa bits, round to nearest
U_FP32 = 2.0 ** -24
EPS = 1e-6                   # GlobalPool's variance epsilon
HEAD_SHAPES = [(64, 64, 128, 101), (64, 64, 128, 128), (64, 64, 128, 2), (16, 16, 32, 101), (48, 16, 128, 101),
               (12, 4, 100, 7), (3, 5, 12, 9), (1, 7, 1, 2)]


# ------------------------------------------------------------------------------------------------------------------
# fp64 references
# ------------------------------------------------------------------------------------------------------------------
def tf32(x: torch.Tensor) -> torch.Tensor:
    """fp64 values of cvt.rna.tf32.f32 applied to fp32(x): nearest at 13 dropped bits, ties away from zero."""
    bits = x.detach().to(torch.float32).contiguous().view(torch.int32)
    return ((bits + 0x1000) & ~0x1FFF).view(torch.float32).double()


def tf32_np(x: np.ndarray) -> np.ndarray:
    """The same rounding computed from the value (frexp), independently of the bit pattern."""
    x = np.asarray(x, np.float32).astype(np.float64)
    m, e = np.frexp(x)                                  # x = m * 2^e, 0.5 <= |m| < 1: 11 significant bits = m * 2^11
    return np.sign(m) * np.floor(np.abs(m) * 2.0 ** 11 + 0.5) * np.exp2(e - 11.0)


def _fold_bn64(bn):
    w, b = bn.weight.detach().double(), bn.bias.detach().double()
    rm, rv = bn.running_mean.detach().double(), bn.running_var.detach().double()
    scale = w / torch.sqrt(rv + bn.eps)
    return scale, b - rm * scale, b.abs() + (rm * scale).abs()          # scale, shift, magnitude of shift


def _tf32_rounding_gap(f, ef):
    """Bound on |tf32(f~) - tf32(f)| over the values f~ within ef of f: 0 where the whole interval lies inside one
    TF32 rounding cell of fp32(f) (both round to the same value), else ef plus both roundings (U_TF32 each, c = 1)
    plus the fp32 rounding of f that the reference's tf32() applies first."""
    a = f.abs()
    slack = ef + U_FP32 * a
    t = (a.to(torch.float32).view(torch.int32) & ~0x1FFF).view(torch.float32).double()      # truncation toward 0
    step = torch.where(t > 0, torch.exp2(torch.floor(torch.log2(torch.where(t > 0, t, torch.ones_like(t)))) - 10),
                       torch.zeros_like(t))
    # rounding boundaries next to a: t + step/2 inside [t, t + step], t + 3 step/2 above, >= step/4 below t
    near = ((a - (t + step / 2)).abs() <= slack) | (t + 1.5 * step - a <= slack) | (a - t + step / 4 <= slack)
    near = near | (slack >= a)                                         # the interval reaches 0
    return torch.where(near, ef + U_TF32 * (2 * a + ef) + U_FP32 * a, torch.zeros_like(a))


def _dense(f, ef, weight, bias, emulate):
    """y = f @ W.T (+ b) with the operand rounding of heads_tail_kernel's mma.sync layers (emulate: features by
    cvt.rna, weights as pack_mma_b) and the bound of the kernel's error on y, given a bound ef of its error on the
    input f: the features whose TF32 rounding may differ from the reference's (_tf32_rounding_gap), fp32 accumulation
    over K exact TF32 products (c = 2), one fp32 rounding of the bias add (c = 1)."""
    W = tf32(weight) if emulate else weight.detach().double()
    y = (tf32(f) if emulate else f) @ W.T
    aw = W.abs()
    err = _tf32_rounding_gap(f, ef) @ aw.T + 2 * W.size(1) * U_FP32 * (f.abs() @ aw.T)
    if bias is not None:
        y = y + bias.detach().double()
        err = err + U_FP32 * y.abs()
    return y, err


def _pool64(z):
    """GlobalPool in fp64 on [n, C, 36] and the bound of heads_tail_kernel's fp32 pooling error: mean and std from
    the shifted sums of d = x - x[cell 0] over 36 cells (c = 2), max exact."""
    mean, mx = z.mean(2), z.amax(2)
    var = ((z - mean.unsqueeze(2)) ** 2).mean(2)
    std = torch.sqrt(var + EPS)
    d = z - z[:, :, :1]
    md, ed2 = d.mean(2), (d * d).mean(2)
    e_mean = 2 * 36 * U_FP32 * d.abs().mean(2) + 2 * U_FP32 * mean.abs()
    e_std = 2 * 36 * U_FP32 * (ed2 + md * md) / std + 2 * U_FP32 * std
    return torch.cat([mean, mx, std], 1), torch.cat([e_mean, torch.zeros_like(mx), e_std], 1)


def heads_tail_ref(pv: torch.Tensor, model, emulate_tf32: bool) -> dict:
    """fp64 PolicyHead / ValueHead after their relu(bn1(conv1)), read from the ChessNet `model` itself.

    pv: [n, pc + vc, 6, 6] (policy channels first), any float dtype.  Returns fp64 log_heads [n, 3, 36], value_logits
    [n, bins], value [n] (expectation over linspace(-1, 1, bins)), pooled_p / pooled_v [n, 3C] (mean | max | std),
    and err_* = the bound of heads_tail_kernel's error on each output (meaningful with emulate_tf32, which rounds the
    dense layers' operands as the kernel does: features by cvt.rna, weights as pack_mma_b)."""
    ph, vh = model.policy_head, model.value_head
    pc = ph.conv1.out_channels
    n = pv.size(0)
    x = pv.detach().double().reshape(n, pv.size(1), 36)
    xp = x[:, :pc]
    fp, efp = _pool64(xp)
    fv, efv = _pool64(x[:, pc:])
    # policy: g = gpool_linear(pooled), p2 = relu(bn2(p + g)), three 1x1 output convs, log-softmax over 36 cells
    g, eg = _dense(fp, efp, ph.gpool_linear.weight, None, emulate_tf32)
    s2, t2, t2mag = _fold_bn64(ph.bn2)
    pre = s2.view(1, -1, 1) * (xp + g.unsqueeze(2))
    p2 = torch.relu(pre + t2.view(1, -1, 1))
    e_p2 = (s2.abs().view(1, -1, 1) * eg.unsqueeze(2)
            + 4 * U_FP32 * (s2.abs().view(1, -1, 1) * (xp.abs() + g.abs().unsqueeze(2)) + t2mag.view(1, -1, 1)))
    wout = torch.stack([ph.out_pos1.weight.detach().double().reshape(-1), ph.out_pos2.weight.detach().double().reshape(-1),
                        ph.out_mark.weight.detach().double().reshape(-1)])
    logits = torch.einsum("hc,ncs->nhs", wout, p2)
    e_logits = (torch.einsum("hc,ncs->nhs", wout.abs(), e_p2)
                + 2 * pc * U_FP32 * torch.einsum("hc,ncs->nhs", wout.abs(), p2))
    lse = torch.logsumexp(logits, 2, keepdim=True)
    log_heads = logits - lse
    # log-softmax is 1-Lipschitz per entry plus the row's largest shift; expf / logf / the 36-term sum in fp32 (c = 4)
    e_log = (e_logits + e_logits.amax(2, keepdim=True)
             + 4 * U_FP32 * (36 + (logits - logits.amax(2, keepdim=True)).abs() + lse.abs()))
    # value: relu(fc1(pooled)), fc2, bucket expectation
    h, eh = _dense(fv, efv, vh.fc1.weight, vh.fc1.bias, emulate_tf32)
    vl, evl = _dense(torch.relu(h), eh, vh.fc2.weight, vh.fc2.bias, emulate_tf32)
    bins = vl.size(1)
    centers = torch.linspace(-1.0, 1.0, bins, dtype=torch.float64, device=vl.device)
    value = (torch.softmax(vl, 1) * centers).sum(1)
    # value = sum p_i c_i moves by sum p_i (c_i - value) dl_i to first order.  Along the way from the reference's
    # logits to the kernel's (each within err_i, D = the row's largest), p_i grows by at most e^(2D) and value moves by
    # at most e^(2D) - 1, which bounds the higher orders.  fp32: expf of l_i - max (2 ulp + the subtraction), the two
    # sums over the bins and the centres -1 + step * k (c = 4).
    p = torch.softmax(vl, 1)
    big_d = evl.amax(1, keepdim=True)
    first = (p * ((centers - value.unsqueeze(1)).abs() + torch.expm1(2 * big_d)) * evl).sum(1)
    e_value = (torch.exp(2 * big_d.squeeze(1)) * first
               + 4 * U_FP32 * (bins + 3 + (vl - vl.amax(1, keepdim=True)).abs().amax(1)) * (p * centers.abs()).sum(1))
    return {"log_heads": log_heads, "value_logits": vl, "value": value, "pooled_p": fp, "pooled_v": fv,
            "err_log_heads": e_log, "err_value_logits": evl, "err_value": e_value}


_DIRS = ((-1, 0), (1, 0), (0, -1), (0, 1))


def combined_logits64(log_heads: torch.Tensor) -> torch.Tensor:
    """[n, 3, 36] log-heads -> fp64 [n, 220] logits in action order: placement (36), movement (cell * 4 + dir; the
    move-from log-prob + the destination's placement log-prob; -inf off the board), mark / capture (36), 4 auxiliary
    actions at 0."""
    lh = log_heads.double()
    n = lh.size(0)
    out = torch.full((n, 220), -math.inf, dtype=torch.float64, device=lh.device)
    out[:, :36] = lh[:, 0]
    for cell in range(36):
        r, c = divmod(cell, 6)
        for d, (dr, dc) in enumerate(_DIRS):
            if 0 <= r + dr < 6 and 0 <= c + dc < 6:
                out[:, 36 + cell * 4 + d] = lh[:, 1, cell] + lh[:, 0, (r + dr) * 6 + c + dc]
    out[:, 180:216] = lh[:, 2]
    out[:, 216:] = 0.0
    return out


def project_priors64(log_heads: torch.Tensor, legal: torch.Tensor):
    """fp64 softmax of the combined logits over each row's legal actions; all 0 for a row with no legal action.
    Returns (priors, combined logits)."""
    comb = combined_logits64(log_heads)
    masked = torch.where(legal, comb, torch.full_like(comb, -math.inf))
    live = legal.any(1, keepdim=True)
    mx = torch.where(live, masked.amax(1, keepdim=True), torch.zeros_like(comb[:, :1]))
    e = torch.where(legal, torch.exp(masked - mx), torch.zeros_like(comb))
    p = e / torch.where(live, e.sum(1, keepdim=True), torch.ones_like(mx))
    return p, comb


def _perturb_bn(model, seed):
    g = torch.Generator().manual_seed(seed)
    for m in model.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            c = m.num_features
            m.running_mean.copy_(torch.randn(c, generator=g) * 0.3)
            m.running_var.copy_(torch.rand(c, generator=g) + 0.5)
            m.weight.data.copy_(torch.rand(c, generator=g) + 0.5)
            m.bias.data.copy_(torch.randn(c, generator=g) * 0.2)
    return model


def _heads_net(pc, vc, mlp, bins, seed, trunk=16):
    from liuzhou_b200.net import ChessNet

    torch.manual_seed(seed)
    model = ChessNet(trunk_channels=trunk, num_blocks=0, policy_channels=pc, value_channels=vc, value_mlp_channels=mlp,
                     value_bucket_bins=bins)
    return _perturb_bn(model, seed).eval()


def _playout_states(n_games, seed, every):
    """Oracle playouts sampled every `every` plies, plus each game's final (terminal) state."""
    out = []
    for game in range(n_games):
        trace = oracle.random_playout(seed, game, 512, want_trace=True)["trace"]
        st = oracle.initial_states(1)
        for ply, a in enumerate(trace):
            if ply % every == 0:
                out.append(st)
            st = oracle.apply_move_scalar(st, int(a))
        out.append(st)
    return concat_states(out)


def _oracle_legal(st) -> np.ndarray:
    n = st["board"].shape[0]
    legal = np.zeros((n, 220), bool)
    for i in range(n):
        legal[i, oracle.legal_actions(st, i)[0]] = True
    return legal


# ------------------------------------------------------------------------------------------------------------------
# CPU: the reference, the projection and the packers
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("pc,vc,mlp,bins", [(64, 64, 128, 101), (3, 5, 12, 9)])
def test_heads_reference_matches_modules_in_fp64(pc, vc, mlp, bins):
    from liuzhou_b200.net import bucket_logits_to_scalar

    model = _heads_net(pc, vc, mlp, bins, seed=pc + vc).double()
    a = torch.randn((32, 16, 6, 6), generator=torch.Generator().manual_seed(1), dtype=torch.float64)
    ph, vh = model.policy_head, model.value_head
    with torch.no_grad():
        pv = torch.cat([ph.act1(ph.bn1(ph.conv1(a))), vh.act1(vh.bn1(vh.conv1(a)))], 1)
        lp = ph(a)
        vl = vh(a)
        pooled = (ph.gpool(pv[:, :pc]), vh.gpool(pv[:, pc:]))
    assert (pv == 0).any() and (pv > 0).any()
    ref = heads_tail_ref(pv, model, emulate_tf32=False)
    for h in range(3):
        assert float((ref["log_heads"][:, h] - lp[h]).abs().max()) <= 1e-12
    assert float((ref["value_logits"] - vl).abs().max()) <= 1e-12
    assert float((ref["value"] - bucket_logits_to_scalar(vl)).abs().max()) <= 1e-12
    assert float((ref["pooled_p"] - pooled[0]).abs().max()) <= 1e-12
    assert float((ref["pooled_v"] - pooled[1]).abs().max()) <= 1e-12


def test_fp64_projection_matches_oracle_projection():
    st = _playout_states(6, 17, every=3)
    legal = _oracle_legal(st)
    n = legal.shape[0]
    no_legal = ~legal.any(1)
    pass_only = legal.any(1) & ~legal[:, :216].any(1)
    assert no_legal.any()                                   # the playouts' terminal states
    g = torch.Generator().manual_seed(4)
    lh = torch.log_softmax(torch.randn((n, 3, 36), generator=g, dtype=torch.float64) * 3, 2)
    p64, _ = project_priors64(lh, torch.from_numpy(legal))
    p32, _ = oracle.project_policy_logits_fast(*(lh[:, h].float().numpy() for h in range(3)), legal)
    assert np.abs(p64.numpy() - p32).max() <= 1e-6
    p = p64.numpy()
    assert (p[~legal] == 0).all() and (p[no_legal] == 0).all()
    assert np.abs(p[~no_legal].sum(1) - 1).max() <= 1e-12
    if pass_only.any():                                     # a state whose only moves are auxiliary actions
        assert np.abs(p[pass_only][:, 216:].sum(1) - 1).max() <= 1e-12


def _mutated(model, what):
    m = copy.deepcopy(model)
    with torch.no_grad():
        if what == "fc2 bias dropped":
            m.value_head.fc2.bias.zero_()
        elif what == "fc1 bias dropped":
            m.value_head.fc1.bias.zero_()
        elif what == "bn2 shift zeroed":
            m.policy_head.bn2.bias.zero_()
            m.policy_head.bn2.running_mean.zero_()
        elif what == "gpool_linear x 0.9":
            m.policy_head.gpool_linear.weight.mul_(0.9)
    return m


@pytest.mark.parametrize("pc,vc,mlp,bins", [(64, 64, 128, 101), (3, 5, 12, 9)])
def test_heads_bound_rejects_wrong_heads(pc, vc, mlp, bins):
    """The bounds the GPU tests hold heads_tail_kernel to are tight enough to fail a kernel that computes a slightly
    different network or decodes the value wrongly."""
    model = _heads_net(pc, vc, mlp, bins, seed=pc * 7 + bins).to(torch.bfloat16)
    vals = _pattern_values(300, pc + vc, seed=bins, device="cpu")
    ref = heads_tail_ref(vals, model, emulate_tf32=True)
    same = _heads_violations(ref, ref["log_heads"], ref["value_logits"], ref["value"])
    assert not any(same.values())
    wrong = {}
    for what in ("fc2 bias dropped", "fc1 bias dropped", "bn2 shift zeroed", "gpool_linear x 0.9"):
        r = heads_tail_ref(vals, _mutated(model, what), emulate_tf32=True)
        wrong[what] = _heads_violations(ref, r["log_heads"], r["value_logits"], r["value"])
    wrong["value negated"] = _heads_violations(ref, ref["log_heads"], ref["value_logits"], -ref["value"])
    wrong["value zero"] = _heads_violations(ref, ref["log_heads"], ref["value_logits"], 0 * ref["value"])
    key = {"fc2 bias dropped": "value_logits", "fc1 bias dropped": "value_logits", "bn2 shift zeroed": "log_heads",
           "gpool_linear x 0.9": "log_heads", "value negated": "value",
           "value zero": "value"}
    missed = {k: v for k, v in wrong.items() if v[key[k]] == 0}
    assert not missed, missed


@pytest.mark.parametrize("n", [1, 7, 8, 9, 192])
@pytest.mark.parametrize("k", [1, 7, 8, 9, 192])
def test_pack_mma_b_layout(n, k):
    """element (nt, ks, lane, j) = tf32(W[nt*8 + lane//4][ks*8 + lane%4 + 4j]), zero padded."""
    from liuzhou_b200.net import pack_mma_b

    rng = np.random.default_rng(n * 1000 + k)
    w = rng.standard_normal((n, k)).astype(np.float32) * np.exp2(rng.integers(-8, 8, (n, k))).astype(np.float32)
    ties = (1.0 + np.array([1, 3, 5, 1, 3], np.float64) * 2.0 ** -11) * np.array([1, 1, 4, -1, -0.5])
    w.reshape(-1)[:min(w.size, ties.size)] = ties[:min(w.size, ties.size)]      # exact ties: away from zero
    got = pack_mma_b(torch.from_numpy(w)).numpy()
    nt, ks = -(-n // 8), -(-k // 8)
    assert got.shape == (nt, ks, 32, 2) and got.dtype == np.float32
    exp = np.zeros((nt, ks, 32, 2))
    wr = tf32_np(w)
    for t in range(nt):
        for s in range(ks):
            for lane in range(32):
                for j in range(2):
                    r, c = t * 8 + lane // 4, s * 8 + lane % 4 + 4 * j
                    if r < n and c < k:
                        exp[t, s, lane, j] = wr[r, c]
    assert np.array_equal(got.astype(np.float64), exp)
    # the ties: 1 + 1/2 step, 1 + 3/2 steps, 4 * (1 + 5/2 steps), their negatives -> one step further from zero
    np.testing.assert_array_equal(tf32_np(ties), [1 + 2 ** -10, 1 + 2 * 2 ** -10, 4 * (1 + 3 * 2 ** -10),
                                                  -(1 + 2 ** -10), -0.5 * (1 + 2 * 2 ** -10)])
    assert torch.equal(tf32(torch.from_numpy(w)), torch.from_numpy(wr))        # the reference's rounding too


def test_pack_conv_weight_layout():
    from liuzhou_b200.net import pack_conv_weight

    w = torch.randn((128, 64, 3, 3), generator=torch.Generator().manual_seed(2))
    got = pack_conv_weight(w)
    assert got.shape == (9, 128, 64) and got.dtype == torch.bfloat16
    for ky in range(3):
        for kx in range(3):
            assert torch.equal(got[ky * 3 + kx], w[:, :, ky, kx].to(torch.bfloat16))
    one = pack_conv_weight(w[:, :, 1:2, 1:2])
    assert one.shape == (1, 128, 64) and torch.equal(one[0], w[:, :, 1, 1].to(torch.bfloat16))


# ------------------------------------------------------------------------------------------------------------------
# GPU: heads_tail_kernel
# ------------------------------------------------------------------------------------------------------------------
def _bf16_step(c: float, k: int) -> torch.Tensor:
    """The bf16 value k representable steps above c (below for k < 0)."""
    return (torch.tensor([c], dtype=torch.bfloat16).view(torch.int16) + k).view(torch.bfloat16).float()


def _pattern_values(n: int, channels: int, seed: int, device) -> torch.Tensor:
    """bf16-representable pv >= 0 [n, channels, 36] with one pattern per (state, channel), every pattern present:
    all zeros; constant at 0.5 / 4 / 30 / 200; near-constant at 1 / 4 / 16 / 48 with 1-3 cells one bf16 step away;
    one hot cell at cell 0 or 35; relu(N(0, s)) for s from 0.1 to 8."""
    g = torch.Generator().manual_seed(seed)
    kinds = [("zero", 0.0)] + [("const", c) for c in (0.5, 4.0, 30.0, 200.0)] + \
            [("near", c) for c in (1.0, 4.0, 16.0, 48.0)] + [("hot", 0), ("hot", 35)] + \
            [("relu", s) for s in (0.1, 0.3, 1.0, 2.0, 4.0, 8.0)]
    rows = n * channels
    out = torch.zeros((rows, 36))
    kind_of = (torch.arange(rows) + int(torch.randint(0, len(kinds), (1,), generator=g))) % len(kinds)
    noise = torch.randn((rows, 36), generator=g)
    for ki, (kind, c) in enumerate(kinds):
        sel = kind_of == ki
        m = int(sel.sum())
        if m == 0:
            continue
        if kind == "const":
            out[sel] = c
        elif kind == "near":
            cells = torch.rand((m, 36), generator=g).argsort(1)[:, :3]
            moved = torch.arange(3) <= (torch.arange(m) % 3).unsqueeze(1)           # 1, 2 or 3 cells
            step = torch.where(torch.rand((m, 1), generator=g) < 0.5, _bf16_step(c, 1), _bf16_step(c, -1))
            block = torch.full((m, 36), c)
            block.scatter_(1, cells, torch.where(moved, step.expand(m, 3), torch.full((m, 3), c)))
            out[sel] = block
        elif kind == "hot":
            out[sel, c] = 3.0
        elif kind == "relu":
            out[sel] = torch.relu(noise[sel] * c)
    return out.to(torch.bfloat16).reshape(n, channels, 36).to(device)


def _pv_tensor(vals: torch.Tensor) -> torch.Tensor:
    n, c, _ = vals.shape
    return vals.reshape(n, c, 6, 6).contiguous(memory_format=torch.channels_last)


def _fused_heads(model):
    from liuzhou_b200.net import FusedHeads

    return FusedHeads(model, tc=False)


def _run_tail(fh, pv, states):
    n = pv.size(0)
    priors = torch.full((n, 220), float("nan"), device=DEV)
    values = torch.full((n,), float("nan"), device=DEV)
    lp1, lp2, lpm, vl = fh.tail(pv, states, priors_out=priors, values_out=values, want_raw=True)
    torch.cuda.synchronize()
    return torch.stack([lp1, lp2, lpm], 1), vl, priors, values


def _heads_violations(ref, log_heads, vl, values) -> dict:
    """Number of elements of each heads output outside the reference's error bound."""
    out = {}
    for name, got in (("log_heads", log_heads), ("value_logits", vl), ("value", values)):
        out[name] = int(((got.double().reshape(ref[name].shape) - ref[name]).abs() > ref["err_" + name]).sum())
    return out


def _check_heads(fh, model, pv, log_heads, vl, values, what):
    ref = heads_tail_ref(pv, model, emulate_tf32=True)
    bad = _heads_violations(ref, log_heads, vl, values)
    ratio = {k: float(((v.double().reshape(ref[k].shape) - ref[k]).abs() / ref["err_" + k]).max())
             for k, v in (("log_heads", log_heads), ("value_logits", vl), ("value", values))}
    assert not any(bad.values()), (what, bad, ratio)


def _check_priors(log_heads, priors, legal, what):
    """Kernel priors vs the fp64 projection of the kernel's own log-heads: the combined logit's fp32 add and
    subtraction of the max, expf (2 ulp) and the fp32 sum over the legal actions (c = 2); a prior below fp32's
    smallest normal number may underflow (the sum is >= 1, so such a prior is < 2^-126)."""
    p64, comb = project_priors64(log_heads, legal)
    live = legal.any(1, keepdim=True)
    mx = torch.where(live, torch.where(legal, comb, torch.full_like(comb, -math.inf)).amax(1, keepdim=True),
                     torch.zeros_like(comb[:, :1]))
    delta = torch.where(legal, U_FP32 * (comb.abs() + (comb - mx).abs() + 2), torch.zeros_like(comb))
    count = legal.sum(1, keepdim=True).double()
    bound = 2 * p64 * (delta + delta.amax(1, keepdim=True) + (count + 1) * U_FP32) + 2.0 ** -126
    diff = (priors.double() - p64).abs()
    assert not (diff > bound).any(), (what, float(diff.max()), float((diff / bound.clamp_min(1e-300)).max()))
    assert (priors[~legal] == 0).all()
    assert (priors[~live.squeeze(1)] == 0).all()
    if live.any():
        sums = priors[live.squeeze(1)].double().sum(1)
        assert float((sums - 1).abs().max()) <= 2 * 220 * U_FP32


def _playout_packed(n, steps, seed):
    from liuzhou_b200 import native

    pb = native.PlayoutBatch(n, seed=seed, device=DEV)
    pb.run(max_steps=steps)
    words, _ = native.legal_masks(pb.packed, scalar_semantics=True)
    return pb.packed, native.mask_words_to_bool(words)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 9, 4737])
def test_pooled_features_exact_through_identity_value_head(n):
    """vc = 40, mlp = bins = 120, fc1 = fc2 = I, zero biases, pv >= 0: value_logits[:, j] is tf32(pooled feature j)
    exactly (mean | max | std of GlobalPool), so the pooled features are checked on their own."""
    model = _heads_net(8, 40, 120, 120, seed=3)
    with torch.no_grad():
        model.value_head.fc1.weight.copy_(torch.eye(120))
        model.value_head.fc2.weight.copy_(torch.eye(120))
        model.value_head.fc1.bias.zero_()
        model.value_head.fc2.bias.zero_()
    model = model.to(DEV, torch.bfloat16)
    fh = _fused_heads(model)
    vals = _pattern_values(n, 48, seed=n, device=DEV)
    _, _, _, vl = fh.tail(_pv_tensor(vals), want_raw=True)
    feat, _ = _pool64(vals[:, 8:].double())
    diff = (vl.double() - feat).abs()
    bound = 2.0 ** -10 * feat.abs() + 1e-7
    bad = diff > bound
    if bad.any():
        s, j = [int(v) for v in bad.nonzero()[0]]
        pytest.fail(f"{int(bad.sum())} of {bad.numel()} pooled features off; state {s} feature {j} "
                    f"({('mean', 'max', 'std')[j // 40]} of channel {j % 40}): kernel {float(vl[s, j])!r}, "
                    f"fp64 {float(feat[s, j])!r}, channel {vals[s, 8 + j % 40].float().tolist()}")


@pytest.mark.gpu
@pytest.mark.parametrize("pc,vc,mlp,bins", HEAD_SHAPES)
def test_heads_tail_kernel_vs_fp64_shapes(pc, vc, mlp, bins):
    model = _heads_net(pc, vc, mlp, bins, seed=pc * 7 + bins).to(DEV, torch.bfloat16)
    fh = _fused_heads(model)
    n = 300
    vals = _pattern_values(n, pc + vc, seed=bins, device=DEV)
    pv = _pv_tensor(vals)
    packed, legal = _playout_packed(n, 25, seed=pc + vc)
    log_heads, vl, priors, values = _run_tail(fh, pv, packed)
    _check_heads(fh, model, pv, log_heads, vl, values, (pc, vc, mlp, bins))
    _check_priors(log_heads, priors, legal, (pc, vc, mlp, bins))


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 7, 8, 9, 4736, 4737, 16384])
def test_heads_tail_kernel_vs_fp64_batch_edges(n):
    """One state, a partial tile, one whole tile, two tiles, one tile per block (148 SMs x 4 blocks x 8), the first
    grid-strided tile, and the product path's chunk."""
    model = _heads_net(64, 64, 128, 101, seed=5).to(DEV, torch.bfloat16)
    fh = _fused_heads(model)
    vals = _pattern_values(n, 128, seed=n, device=DEV)
    g = torch.Generator(device=DEV).manual_seed(n)
    vals = torch.where(torch.rand(vals.shape, generator=g, device=DEV) < 0.5, vals,
                       torch.relu(torch.randn(vals.shape, generator=g, device=DEV)).to(torch.bfloat16))
    pv = _pv_tensor(vals)
    packed, legal = _playout_packed(n, 40, seed=n)
    log_heads, vl, priors, values = _run_tail(fh, pv, packed)
    _check_heads(fh, model, pv, log_heads, vl, values, n)
    _check_priors(log_heads, priors, legal, n)


@pytest.mark.gpu
def test_heads_tail_priors_on_oracle_states():
    """Legal sets from the oracle: playout states, terminal states (no legal action: all-zero rows)."""
    model = _heads_net(64, 64, 128, 101, seed=8).to(DEV, torch.bfloat16)
    fh = _fused_heads(model)
    from liuzhou_b200 import native

    st = _playout_states(4, 23, every=2)
    legal = torch.from_numpy(_oracle_legal(st)).to(DEV)
    n = legal.size(0)
    assert not legal.any(1).all()
    packed = native.pack_states(to_torch(st, DEV))
    pv = _pv_tensor(_pattern_values(n, 128, seed=9, device=DEV))
    log_heads, vl, priors, values = _run_tail(fh, pv, packed)
    _check_heads(fh, model, pv, log_heads, vl, values, "oracle states")
    _check_priors(log_heads, priors, legal, "oracle states")


@pytest.mark.gpu
def test_heads_tail_kernel_on_product_activations():
    """pv from the default ChessNet's trunk kernel on self-play positions at several depths."""
    from liuzhou_b200 import native
    from liuzhou_b200.net import ChessNet, InferenceNet
    from liuzhou_b200.tree import encode_inputs

    torch.manual_seed(12)
    net = InferenceNet(_perturb_bn(ChessNet(), 12), DEV)
    assert net.path == "trunk"
    n = 16384
    pb = native.PlayoutBatch(n, seed=31, device=DEV)
    for steps in (0, 10, 40, 120):
        pb.run(max_steps=steps)
        x = encode_inputs(pb.packed, "bf16_nhwc", out=net.new_input(n))
        pv = net._trunk_heads_conv(x)
        words, _ = native.legal_masks(pb.packed, scalar_semantics=True)
        log_heads, vl, priors, values = _run_tail(net.heads, pv, pb.packed)
        _check_heads(net.heads, net.model, pv, log_heads, vl, values, steps)
        _check_priors(log_heads, priors, native.mask_words_to_bool(words), steps)


@pytest.mark.gpu
def test_heads_tail_refusals_and_empty_batch():
    from liuzhou_b200._lib import check, i64, lib, ptr, stream_ptr

    model = _heads_net(64, 64, 128, 101, seed=1).to(DEV, torch.bfloat16)
    fh = _fused_heads(model)
    t = fh._t
    n = 16
    pv = _pv_tensor(_pattern_values(n, 128, seed=1, device=DEV))
    packed, _ = _playout_packed(n, 5, seed=1)
    priors = torch.full((n, 220), 7.0, device=DEV)
    values = torch.full((n,), 7.0, device=DEV)

    def call(n=n, pc=64, vc=64, mlp=128, bins=101, pv_addr=pv.data_ptr(), states=packed, priors=priors):
        return lib().lzb_heads_tail(ctypes.c_void_p(pv_addr), i64(n), ctypes.c_int32(pc), ctypes.c_int32(vc),
                                    ctypes.c_int32(mlp), ctypes.c_int32(bins), ptr(t["wgl_t"]), ptr(t["bn2_scale"]),
                                    ptr(t["bn2_shift"]), ptr(t["wout"]), ptr(t["wfc1_t"]), ptr(t["bfc1"]),
                                    ptr(t["wfc2_t"]), ptr(t["bfc2"]), ptr(states), ptr(priors), ptr(values),
                                    ptr(None), ptr(None), stream_ptr(DEV))

    bad_calls = [dict(pc=0), dict(pc=65, vc=63), dict(vc=0, pc=64), dict(vc=65, pc=63), dict(bins=1), dict(bins=129),
                 dict(mlp=0), dict(mlp=129), dict(pc=60, vc=62), dict(pc=3, vc=4), dict(pv_addr=pv.data_ptr() + 2),
                 dict(states=None)]
    for kw in bad_calls:
        with pytest.raises(RuntimeError):
            check(call(**kw))
    check(call(n=0))                                          # an empty batch is a no-op
    torch.cuda.synchronize()
    assert bool((priors == 7.0).all()) and bool((values == 7.0).all())
    check(call())
    torch.cuda.synchronize()
    assert not bool((values == 7.0).any())


# ------------------------------------------------------------------------------------------------------------------
# GPU: bn_relu_kernel
# ------------------------------------------------------------------------------------------------------------------
def _round_bf16_64(y: torch.Tensor) -> torch.Tensor:
    """Round fp64 values to bf16 once (nearest, ties to even), returned as fp64."""
    ulp = bf16_ulp(y)
    return torch.where(ulp > 0, torch.round(y / torch.where(ulp > 0, ulp, torch.ones_like(ulp))) * ulp, y)


def _expect_bf16(got: torch.Tensor, y64: torch.Tensor, what):
    """got == bf16(y64), or 1 bf16 step away where the kernel's fp32 result sits exactly on a bf16 tie."""
    exp = _round_bf16_64(y64)
    g = got.double()
    tie = (y64.float().view(torch.int32) & 0xFFFF) == 0x8000
    off = g != exp
    assert not (off & ~tie).any(), (what, int((off & ~tie).sum()))
    assert not (off & ((g - exp).abs() > bf16_ulp(torch.maximum(g.abs(), exp.abs())))).any(), what


@pytest.mark.gpu
@pytest.mark.parametrize("rows", [1, 7, 36 * 1024])
@pytest.mark.parametrize("channels", [8, 24, 40, 128, 256])
def test_bn_relu_kernel_vs_fp64(channels, rows):
    from liuzhou_b200._lib import check, i64, lib, ptr, stream_ptr

    g = torch.Generator().manual_seed(channels * 100 + rows)
    u = (torch.randn((rows, channels), generator=g) * 2).to(torch.bfloat16).to(DEV)
    v = (torch.randn((rows, channels), generator=g) * 2).to(torch.bfloat16).to(DEV)
    scale = (torch.rand((channels,), generator=g) * 2 - 0.5).to(DEV)
    shift = torch.randn((channels,), generator=g).to(DEV)
    for variant in ("act", "sum+act", "act of sum"):
        guard = 3                                      # rows past the end must stay untouched
        act = torch.full((rows + guard, channels), -5.0, dtype=torch.bfloat16, device=DEV)
        ssum = torch.full((rows + guard, channels), -5.0, dtype=torch.bfloat16, device=DEV)
        vv = None if variant == "act" else v
        out_sum = ssum if variant == "sum+act" else None
        check(lib().lzb_bn_relu_bf16(ptr(u), ptr(vv), ptr(scale), ptr(shift), i64(rows), ctypes.c_int32(channels),
                                     ptr(out_sum), ptr(act), stream_ptr(DEV)))
        torch.cuda.synchronize()
        x = u if vv is None else (u.float() + v.float()).bfloat16()
        if variant == "sum+act":
            assert torch.equal(ssum[:rows], x)
        assert bool((ssum[rows:] == -5.0).all() if variant == "sum+act" else (ssum == -5.0).all())
        assert bool((act[rows:] == -5.0).all())
        y64 = torch.relu(x.double() * scale.double() + shift.double())
        _expect_bf16(act[:rows], y64, (variant, channels, rows))


@pytest.mark.gpu
def test_bn_relu_refusals():
    from liuzhou_b200._lib import check, i64, lib, ptr, stream_ptr

    u = torch.zeros((64, 32), dtype=torch.bfloat16, device=DEV)
    act = torch.empty_like(u)
    scale = torch.ones((40,), device=DEV)
    shift = torch.zeros((40,), device=DEV)

    def call(c=32, u_addr=u.data_ptr(), act_addr=act.data_ptr(), shift_addr=shift.data_ptr()):
        return lib().lzb_bn_relu_bf16(ctypes.c_void_p(u_addr), None, ptr(scale), ctypes.c_void_p(shift_addr), i64(8),
                                      ctypes.c_int32(c), None, ctypes.c_void_p(act_addr), stream_ptr(DEV))

    for kw in (dict(c=12), dict(c=0), dict(c=30), dict(u_addr=u.data_ptr() + 8), dict(act_addr=act.data_ptr() + 2),
               dict(shift_addr=shift.data_ptr() + 4)):
        with pytest.raises(RuntimeError):
            check(call(**kw))
    check(call())
