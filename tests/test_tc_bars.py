"""CPU: the split-bf16 gradient bars of the tensor-core tests sit between the two arithmetics they have to tell apart.

Each tightened test's gradient is recomputed here in fp64 with every tensor-core product's operands rounded the way the
kernels round them: fp32 inputs, split into bf16 hi + lo, products accumulated in fp64, in three arithmetics:
    x3     hi.hi + hi.lo + lo.hi   (NPF_PREC_BF16X3)
    drop1  hi.hi + hi.lo           (a kernel that lost one correction product)
    bf16   hi.hi                   (NPF_PREC_BF16)
Every bf16x3 bar must be at least 5x the emulated x3 error (room for the fp32 accumulation and ordering of the device) and
at most 1/5 of the emulated drop1 error (so a lost correction product fails the test).  A later change that loosens a bar
past the second line, or tightens it below the first, fails here without a GPU."""
import math

import pytest
import torch
import torch.nn.functional as F

import test_gpu_ops as ops_t
import test_gpu_tc as tc_t
import test_gpu_tc_paths as paths_t

_mode = ["x3"]


def _split(x):
    xf = x.float()
    hi = xf.bfloat16().float()
    lo = (xf - hi).bfloat16().float()
    return hi.double(), lo.double()


def mm(a, b):
    """a @ b (batched) with both operands rounded as the current arithmetic `_mode[0]` rounds them."""
    ah, al = _split(a)
    bh, bl = _split(b)
    out = ah @ bh
    if _mode[0] in ("x3", "drop1"):
        out = out + ah @ bl
    if _mode[0] == "x3":
        out = out + al @ bh
    return out


class _MM(torch.autograd.Function):
    """a @ b whose forward and both backward products are tensor-core products."""

    @staticmethod
    def forward(ctx, a, b):
        ctx.save_for_backward(a, b)
        return mm(a, b)

    @staticmethod
    def backward(ctx, g):
        a, b = ctx.saved_tensors
        return mm(g, b.transpose(-1, -2)), mm(a.transpose(-1, -2), g)


def _g(*shape, seed=0, scale=1.0):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed), dtype=torch.float64) * scale


def _fp32(t):
    return t.float().double()


def l2(a, b):
    return ((a - b).norm() / b.norm()).item()


def maxrel(a, b):
    return ((a - b).abs().max() / b.abs().max()).item()


# ------------------------------------------------------------------------------------------------ emulations
def emu_fused_linear_backward(M=1000):
    """test_tc_fused_linear_backward: dX = (dY W) (.) (X > 0), dW = dY^T X."""
    dY, W, X = _fp32(_g(M, 128, seed=1)), _fp32(_g(128, 128, seed=2, scale=128 ** -0.5)), _fp32(torch.relu(_g(M, 128, seed=3)))
    return max(l2(mm(dY, W) * (X > 0), (dY @ W) * (X > 0)), l2(mm(dY.t(), X), dY.t() @ X))


def emu_chain_bwd(L=8, M=4099):
    """test_tc_mlp_chain_bwd_entry: the gradient image is re-split after every layer."""
    Ws = [_fp32(_g(128, 128, seed=10 + l, scale=128 ** -0.5)) for l in range(L)]
    Xs = [_g(M, 128, seed=1)]
    for l in range(L - 1):
        Xs.append(torch.relu(Xs[-1] @ Ws[l].t() + 0.1 * _g(128, seed=40 + l)))
    Xs = [_fp32(x) for x in Xs]
    dz = dze = _fp32(_g(M, 128, seed=2))
    errs = []
    for l in range(L - 1, -1, -1):
        errs.append(l2(mm(dze.t(), Xs[l]), dz.t() @ Xs[l]))
        dz, dze = dz @ Ws[l], mm(dze.float().double(), Ws[l])
        if l > 0:
            dz, dze = dz * (Xs[l] > 0), dze * (Xs[l] > 0)
    return max(errs + [l2(dze, dz)])


def emu_single_linear(M=513, K=128, N=128):
    """test_tc_single_linear_localised: dx = go W, dW = go^T x (max-rel)."""
    x, W, go = _fp32(_g(M, K, seed=1)), _fp32(_g(N, K, seed=2, scale=K ** -0.5)), _fp32(_g(M, N, seed=4))
    return max(maxrel(mm(go, W), go @ W), maxrel(mm(go.t(), x), go.t() @ x))


def _attn(q, k, v, H, D, prod):
    heads = lambda t: t.view(t.shape[0], t.shape[1], H, D).transpose(1, 2)
    s = heads(q) @ heads(k).transpose(-1, -2) / math.sqrt(D)      # logits: six-term split, fp32-accurate
    return prod(s.softmax(-1), heads(v)).transpose(1, 2).reshape(q.shape[0], q.shape[1], H * D)


def emu_attention(B=2, Tq=128, Tk=128, H=8, D=16):
    """test_tc_attention_forward gradients: P V forward; dP = dO V^T, dV = P^T dO, dQ = dS K, dK = dS^T Q backward."""
    q, k, v = _fp32(_g(B, Tq, H * D, seed=1)), _fp32(_g(B, Tk, H * D, seed=2)), _fp32(_g(B, Tk, H * D, seed=3))
    go = _fp32(_g(B, Tq, H * D, seed=9))
    grads = {}
    for name, prod in (("ref", torch.matmul), ("emu", None)):
        r = [t.clone().requires_grad_(True) for t in (q, k, v)]
        if prod is None:
            heads = lambda t: t.view(B, t.shape[1], H, D).transpose(1, 2)
            # value: the fp32-accurate logits; gradient: through the split products dQ = dS K, dK = dS^T Q
            s = _MM.apply(heads(r[0]), heads(r[1]).transpose(-1, -2)) / math.sqrt(D)
            s = (heads(r[0]) @ heads(r[1]).transpose(-1, -2) / math.sqrt(D)).detach() + (s - s.detach())
            y = _MM.apply(s.softmax(-1), heads(r[2])).transpose(1, 2).reshape(B, Tq, H * D)
        else:
            y = _attn(*r, H, D, prod)
        y.backward(go)
        grads[name] = [t.grad for t in r]
    return max(l2(a, b) for a, b in zip(grads["emu"], grads["ref"]))


def emu_resblock(B=2, L=384):
    """test_resblock1d_fused gradients: the pointwise product and both of its backward products on tensor cores."""
    x, wd, bd = _fp32(_g(B, L, 128, seed=1)), _fp32(_g(128, 1, 11, seed=2, scale=0.3)), _fp32(_g(128, seed=3))
    wp, bp = _fp32(_g(128, 128, 1, seed=4, scale=128 ** -0.5)), _fp32(_g(128, seed=5))
    go = _fp32(_g(B, L, 128, seed=99))
    grads = {}
    for name, prod in (("ref", torch.matmul), ("emu", _MM.apply)):
        r = [t.clone().requires_grad_(True) for t in (x, wd, bd, wp, bp)]
        o = F.conv1d(torch.relu(r[0]).transpose(1, 2), r[1], r[2], padding=5, groups=128).transpose(1, 2) + r[0]
        y = prod(o, r[3].view(128, 128).t()) + r[4]
        y.backward(go)
        grads[name] = [t.grad for t in r]
    return max(maxrel(a, b) for a, b in zip(grads["emu"], grads["ref"]))


def emu_setconv(B=3, K=296, Q=128, C=128, N=128, sigma=0.012):
    """test_setconv (C = 128, regular grid): the weighted sum of values and the resizer on tensor cores."""
    gen = torch.Generator().manual_seed(K * 7 + Q)
    keys = torch.linspace(-1.5, 1.5, K).double().view(1, 1, K)
    queries = _fp32((torch.rand(B, Q, 1, generator=gen, dtype=torch.float64) * 2 - 1))
    values, W, b = _fp32(_g(B, K, C, seed=3)), _fp32(_g(N, C + 1, seed=4, scale=(C + 1) ** -0.5)), _fp32(_g(N, seed=5))
    a = -((keys - queries) / sigma) ** 2
    w, dens = torch.softmax(a, -1), torch.exp(a).sum(-1, keepdim=True)
    go = _fp32(_g(B, Q, N, seed=99))
    grads = {}
    for name, prod in (("ref", torch.matmul), ("emu", _MM.apply)):
        r = [t.clone().requires_grad_(True) for t in (values, W, b)]
        feat = prod(w, r[0])
        y = prod(feat, r[1][:, :C].t()) + dens * r[1][:, C] + r[2]
        y.backward(go)
        grads[name] = [t.grad for t in r]
    return max(maxrel(a_, b_) for a_, b_ in zip(grads["emu"], grads["ref"]))


CASES = {   # tightened test -> (its bf16x3 gradient bar, emulation at its shapes)
    "test_tc_fused_linear_backward": (lambda: tc_t.GBARS["bf16x3"], emu_fused_linear_backward),
    "test_tc_mlp_chain_bwd_entry": (lambda: tc_t.CHAIN_GBARS["bf16x3"], emu_chain_bwd),
    "test_tc_single_linear_localised": (lambda: tc_t.GMAX["bf16x3"], emu_single_linear),
    "test_tc_attention_forward": (lambda: tc_t.ABARS["bf16x3"], emu_attention),
    "test_resblock1d_fused": (lambda: ops_t.TC_GTOL["bf16x3"], emu_resblock),
    "test_setconv": (lambda: ops_t.TC_GTOL["bf16x3"], emu_setconv),
    "test_resblock1d_bwd_accumulates": (lambda: paths_t.RB_GTOL, emu_resblock),
}


@pytest.mark.parametrize("test", sorted(CASES))
def test_bf16x3_bar_separates_split_from_dropped_product(test):
    bar_fn, emu = CASES[test]
    bar = bar_fn()
    errs = {}
    for mode in ("x3", "drop1"):
        _mode[0] = mode
        try:
            errs[mode] = emu()
        finally:
            _mode[0] = "x3"
    assert bar >= 5 * errs["x3"], f"{test}: bar {bar:.1e} is within 5x of the split-bf16 error {errs['x3']:.2e}"
    assert bar <= errs["drop1"] / 5, f"{test}: bar {bar:.1e} would pass a dropped correction product (error {errs['drop1']:.2e})"
