"""-m gpu: tensor-core paths that whole models reach but the op tests above did not, and a check that the split-bf16 mode
really is split-bf16.

* Two-mode check: every kernel that exists in both tensor-core modes runs the same inputs in bf16 and in bf16x3.  The
  split (hi.hi + hi.lo + lo.hi) must be at least 20x closer to fp64 than one bf16 product; a kernel that lost a
  correction product is only ~1.3x closer.  The check sets its own scale, so it holds whatever the inputs.
* C ABI edge cases: operands whose rows are not 16-byte aligned (the scalar-load instantiations), outputs filled with
  NaN so that a row or column the kernel skips shows up, `+=` outputs that start non-zero, and NULL optional outputs.
"""
import ctypes
import math

import pytest
import torch
import torch.nn.functional as F

from _util import rel_err
from test_gpu_tc import CHAIN_GBARS, GBARS, attn_ref, l2_rel

pytestmark = pytest.mark.gpu
PREC = {"bf16": 1, "bf16x3": 2}
RB_GTOL = 5e-5   # npf_resblock1d_bwd gradients, max-rel (the bar of test_gpu_ops.py::test_resblock1d_fused)


@pytest.fixture(scope="module")
def cabi():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    import npf_b200
    from npf_b200 import _cabi
    yield _cabi
    npf_b200.set_precision("fp32")


def _g(*shape, seed=0, scale=1.0):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed), dtype=torch.float64) * scale


def _c(t):
    return t.float().cuda().contiguous()


def _st():
    return torch.cuda.current_stream().cuda_stream


def _arr(ts):
    return (ctypes.c_void_p * len(ts))(*[None if t is None else t.data_ptr() for t in ts])


# ------------------------------------------------------------------------------------------------ two-mode check
def _linear_case(cabi, kernel, pr, M=1000, K=128, N=128):
    """(device results, fp64 references) of one linear-layer entry point at precision code `pr`."""
    X, W, b, dY = _g(M, K, seed=1), _g(N, K, seed=2, scale=K ** -0.5), _g(N, seed=3), _g(M, N, seed=4)
    Xr = torch.relu(X)            # the layer input of a backward: post-ReLU, the mask source
    Xc, Wc, bc, dYc, Xrc = _c(X), _c(W), _c(b), _c(dY), _c(Xr)   # held: the kernels read them after call() returns
    st = _st()
    if kernel == "linear_fwd":
        Y = torch.full((M, N), float("nan"), device="cuda")
        cabi.call("npf_linear_fwd", Xc.data_ptr(), K, Wc.data_ptr(), K, bc.data_ptr(), Y.data_ptr(), N, M, K, N, 0, 0, 0, 0, pr, st)
        return [Y], [X @ W.t() + b]
    if kernel == "linear_bwd_data":
        dX = torch.full((M, K), float("nan"), device="cuda")
        cabi.call("npf_linear_bwd_data", dYc.data_ptr(), N, Wc.data_ptr(), K, dX.data_ptr(), K, M, K, N, 0, 0, 0, pr, st)
        return [dX], [dY @ W]
    if kernel == "linear_bwd_weight":
        dW = torch.zeros(N, K, device="cuda")
        cabi.call("npf_linear_bwd_weight", dYc.data_ptr(), N, Xrc.data_ptr(), K, dW.data_ptr(), K, 0, M, K, N, 0, 0, 0, 0, pr, st)
        return [dW], [dY.t() @ Xr]
    if kernel == "linear_bwd_fused":
        dX, dW = torch.full((M, K), float("nan"), device="cuda"), torch.zeros(N, K, device="cuda")
        cabi.call("npf_linear_bwd", dYc.data_ptr(), N, Xrc.data_ptr(), K, Wc.data_ptr(), K, dX.data_ptr(), K, dW.data_ptr(), K,
                  0, M, K, N, 16, pr, st)
        return [dX, dW], [(dY @ W) * (Xr > 0), dY.t() @ Xr]
    raise ValueError(kernel)


def _chain_case(cabi, kernel, pr, L=3, M=1000):
    Ws = [_g(128, 128, seed=10 + l, scale=128 ** -0.5) for l in range(L)]
    bs = [_g(128, seed=30 + l) for l in range(L)]
    X = _g(M, 128, seed=1)
    st = _st()
    if kernel == "chain_fwd":
        Ys = [torch.full((M, 128), float("nan"), device="cuda") for _ in range(L)]
        Xc, Wc, bc = _c(X), [_c(w) for w in Ws], [_c(b) for b in bs]
        cabi.call("npf_mlp_chain_fwd", Xc.data_ptr(), 128, _arr(Wc), _arr(bc), _arr(Ys), L, M, 128, 0, (1 << (L - 1)) - 1, pr, st)
        h, refs = X, []
        for l in range(L):
            h = h @ Ws[l].t() + bs[l]
            if l < L - 1:
                h = torch.relu(h)
            refs.append(h)
        return Ys[-1:], refs[-1:]
    if kernel == "chain_bwd":
        Xs = [torch.relu(X)]
        for l in range(L - 1):
            Xs.append(torch.relu(Xs[-1] @ Ws[l].t() + 0.1 * _g(128, seed=40 + l)))
        dY = _g(M, 128, seed=2)
        dz, dWr = dY, [None] * L
        for l in range(L - 1, -1, -1):
            dWr[l] = dz.t() @ Xs[l]
            dz = dz @ Ws[l]
            if l > 0:
                dz = dz * (Xs[l] > 0)
        dX = torch.full((M, 128), float("nan"), device="cuda")
        dW = [torch.zeros(128, 128, device="cuda") for _ in range(L)]
        Xc, Wc, dYc = [_c(x) for x in Xs], [_c(w) for w in Ws], _c(dY)
        cabi.call("npf_mlp_chain_bwd", dYc.data_ptr(), 128, _arr(Xc), _arr(Wc), dX.data_ptr(), 128, _arr(dW), None, L, M, 128, 0, pr, st)
        return [dX] + dW, [dz] + dWr
    raise ValueError(kernel)


def _attn_case(kernel, prec, B=2, Tq=130, Tk=150, H=4, D=16):
    import npf_b200
    npf_b200.set_precision(prec)
    q, k, v = _g(B, Tq, H * D, seed=1), _g(B, Tk, H * D, seed=2), _g(B, Tk, H * D, seed=3)
    r = [t.clone().requires_grad_(True) for t in (q, k, v)]
    yr = attn_ref(*r, H, D, D)
    c = [_c(t).requires_grad_(True) for t in (q, k, v)]
    yc = npf_b200.ops.xattn(*c, H, 1.0 / math.sqrt(D))
    if kernel == "attn_fwd":
        return [yc], [yr]
    go = _g(*yr.shape, seed=9)
    yr.backward(go)
    yc.backward(_c(go))
    return [t.grad for t in c], [t.grad for t in r]


@pytest.mark.parametrize("kernel", ["linear_fwd", "linear_bwd_data", "linear_bwd_weight", "linear_bwd_fused", "chain_fwd", "chain_bwd",
                                    "attn_fwd", "attn_bwd"])
def test_split_bf16_beats_bf16(cabi, kernel):
    """err(bf16x3) * 20 <= err(bf16), per output, for the same inputs through the same entry point."""
    errs = {}
    for prec in ("bf16", "bf16x3"):
        if kernel.startswith("linear"):
            outs, refs = _linear_case(cabi, kernel, PREC[prec])
        elif kernel.startswith("chain"):
            outs, refs = _chain_case(cabi, kernel, PREC[prec])
        else:
            outs, refs = _attn_case(kernel, prec)
        torch.cuda.synchronize()
        assert all(torch.isfinite(o).all() for o in outs), prec
        errs[prec] = [l2_rel(o, r) for o, r in zip(outs, refs)]
    for i, (e3, e1) in enumerate(zip(errs["bf16x3"], errs["bf16"])):
        assert e3 * 20 <= e1, f"{kernel} output {i}: bf16x3 {e3:.3e} vs bf16 {e1:.3e}"


# ------------------------------------------------------------------------------------------------ unaligned operands
def _strided(rows, cols, layout, fill):
    """A [rows, cols] view that is NOT 16-byte aligned row by row, in a buffer filled with `fill`: 'ld+1' (leading
    dimension cols + 1) or 'offset' (contiguous rows, base one float past a 16-byte boundary).  Returns (buffer, view, ld)."""
    if layout == "ld+1":
        buf = torch.full((rows * (cols + 1),), fill, device="cuda")
        return buf, buf.view(rows, cols + 1)[:, :cols], cols + 1
    buf = torch.full((rows * cols + 1,), fill, device="cuda")
    return buf, buf[1:].view(rows, cols), cols


def _outside(buf, view):
    """The entries of `buf` that `view` does not cover."""
    keep = torch.ones(buf.numel(), dtype=torch.bool, device=buf.device)
    idx = torch.arange(view.numel(), device=buf.device).view(view.shape)
    keep[view.storage_offset() + (idx // view.shape[1]) * view.stride(0) + idx % view.shape[1]] = False
    return buf[keep]


@pytest.mark.parametrize("prec", ["bf16x3", "bf16"])
@pytest.mark.parametrize("layout", ["ld+1", "offset"])
@pytest.mark.parametrize("M,K,N", [(300, 128, 128), (77, 64, 32)])
def test_linear_fwd_unaligned(cabi, prec, layout, M, K, N):
    """npf_linear_fwd with X and Y rows not 16-byte aligned (scalar-load instantiation of the tensor-core kernel), bias,
    the rank-1 term u (x) w2 with w2 a strided column, relu on input and output; nothing outside Y is written."""
    X, W, b, u = _g(M, K, seed=1), _g(N, K + 1, seed=2, scale=K ** -0.5), _g(N, seed=3), _g(M, seed=4)
    _, Xv, ldx = _strided(M, K, layout, 0.0)
    Xv.copy_(X.float())
    Ybuf, Yv, ldy = _strided(M, N, layout, float("nan"))
    Wc, bc, uc = _c(W), _c(b), _c(u)
    cabi.call("npf_linear_fwd", Xv.data_ptr(), ldx, Wc.data_ptr(), K + 1, bc.data_ptr(), Yv.data_ptr(), ldy, M, K, N, 1 | 2,
              uc.data_ptr(), Wc.data_ptr() + 4 * K, K + 1, PREC[prec], _st())
    torch.cuda.synchronize()
    ref = torch.relu(torch.relu(X) @ W[:, :K].t() + u[:, None] * W[:, K] + b)
    assert torch.isfinite(Yv).all()
    assert rel_err(Yv, ref) < {"bf16x3": 1e-4, "bf16": 1e-2}[prec], rel_err(Yv, ref)
    assert torch.isnan(_outside(Ybuf, Yv)).all()


@pytest.mark.parametrize("prec", ["bf16x3", "bf16"])
@pytest.mark.parametrize("layout", ["ld+1", "offset"])
@pytest.mark.parametrize("M,K,N", [(300, 128, 128), (77, 32, 64)])
def test_linear_bwd_data_unaligned(cabi, prec, layout, M, K, N):
    """npf_linear_bwd_data with dY, dX and the relu-mask source not 16-byte aligned, W with a 16-byte-misaligned row
    stride (the transposed staging's scalar loads); nothing outside dX is written."""
    dY, W, Xm = _g(M, N, seed=1), _g(N, K + 1, seed=2, scale=N ** -0.5), _g(M, K, seed=3)
    _, dYv, lddy = _strided(M, N, layout, 0.0)
    dYv.copy_(dY.float())
    _, Xv, ldm = _strided(M, K, layout, 0.0)
    Xv.copy_(Xm.float())
    dXbuf, dXv, lddx = _strided(M, K, layout, float("nan"))
    Wc = _c(W)
    cabi.call("npf_linear_bwd_data", dYv.data_ptr(), lddy, Wc.data_ptr(), K + 1, dXv.data_ptr(), lddx, M, K, N, Xv.data_ptr(), ldm, 0,
              PREC[prec], _st())
    torch.cuda.synchronize()
    ref = (dY @ W[:, :K]) * (Xm.float().double() > 0)
    assert torch.isfinite(dXv).all()
    assert l2_rel(dXv, ref) < GBARS[prec], l2_rel(dXv, ref)
    assert (dXv[Xv <= 0] == 0).all()
    assert torch.isnan(_outside(dXbuf, dXv)).all()


@pytest.mark.parametrize("prec", ["bf16x3", "bf16"])
@pytest.mark.parametrize("L,M", [(3, 300), (2, 64)])
def test_mlp_chain_bwd_unaligned_weights(cabi, prec, L, M):
    """npf_mlp_chain_bwd with every W_l and dW_l one float past a 16-byte boundary (scalar weight staging, scalar dW
    flush), dW / db accumulated into non-zero buffers, dX NaN-filled."""
    Ws = [_g(128, 128, seed=10 + l, scale=128 ** -0.5) for l in range(L)]
    Xs = [_g(M, 128, seed=1)]
    for l in range(L - 1):
        Xs.append(torch.relu(Xs[-1] @ Ws[l].t() + 0.1 * _g(128, seed=40 + l)))
    dY = _g(M, 128, seed=2)
    dW0 = [_g(128, 128, seed=60 + l) for l in range(L)]
    db0 = [_g(128, seed=80 + l) for l in range(L)]
    dz, dWr, dbr = dY, [None] * L, [None] * L
    for l in range(L - 1, -1, -1):
        dWr[l], dbr[l] = dz.t() @ Xs[l], dz.sum(0)
        dz = dz @ Ws[l]
        if l > 0:
            dz = dz * (Xs[l] > 0)
    Wbuf = torch.zeros(L * 128 * 128 + 1, device="cuda")
    dWbuf = torch.zeros(L * 128 * 128 + 1, device="cuda")
    Wc = [Wbuf[1 + l * 16384:1 + (l + 1) * 16384].view(128, 128) for l in range(L)]
    dWc = [dWbuf[1 + l * 16384:1 + (l + 1) * 16384].view(128, 128) for l in range(L)]
    for l in range(L):
        Wc[l].copy_(Ws[l].float())
        dWc[l].copy_(dW0[l].float())
    Xc, dbc, dYc = [_c(x) for x in Xs], [_c(b) for b in db0], _c(dY)
    dX = torch.full((M, 128), float("nan"), device="cuda")
    cabi.call("npf_mlp_chain_bwd", dYc.data_ptr(), 128, _arr(Xc), _arr(Wc), dX.data_ptr(), 128, _arr(dWc), _arr(dbc), L, M, 128, 0,
              PREC[prec], _st())
    torch.cuda.synchronize()
    assert torch.isfinite(dX).all() and torch.isfinite(dWbuf).all()
    assert l2_rel(dX, dz) < CHAIN_GBARS[prec], ("dX", l2_rel(dX, dz))
    for l in range(L):
        e = l2_rel(dWc[l] - _c(dW0[l]), dWr[l])
        assert e < CHAIN_GBARS[prec], (f"dW{l}", e)
        e = l2_rel(dbc[l] - _c(db0[l]), dbr[l])
        assert e < CHAIN_GBARS[prec], (f"db{l}", e)
    assert dWbuf[0].item() == 0.0


# ------------------------------------------------------------------------------------------------ npf_resblock1d_bwd contract
@pytest.mark.parametrize("with_bias_grads", [True, False])
@pytest.mark.parametrize("B,L", [(2, 384), (3, 100)])
def test_resblock1d_bwd_accumulates(cabi, B, L, with_bias_grads):
    """npf_resblock1d_bwd: dX overwritten (NaN-filled before), dWdw / dWpw (and dbdw / dbpw when given) ADDED to non-zero
    buffers; with dbdw = dbpw = NULL the weight gradients are unchanged."""
    C, k = 128, 11
    x, wd, bd = _g(B, L, C, seed=1), _g(C, 1, k, seed=2, scale=0.3), _g(C, seed=3)
    wp, bp = _g(C, C, seed=4, scale=C ** -0.5), _g(C, seed=5)
    r = [t.clone().requires_grad_(True) for t in (x, wd, bd, wp, bp)]
    o = F.conv1d(torch.relu(r[0]).transpose(1, 2), r[1], r[2], padding=k // 2, groups=C).transpose(1, 2) + r[0]
    y = o @ r[3].t() + r[4]
    dY = _g(B, L, C, seed=6)
    y.backward(dY)
    acc0 = [_g(C, k, seed=7), _g(C, seed=8), _g(C, C, seed=9), _g(C, seed=10)]
    dWd, dbd, dWp, dbp = [_c(t) for t in acc0]
    dX = torch.full((B, L, C), float("nan"), device="cuda")
    xc, wdc, bdc, wpc, dYc = _c(x), _c(wd), _c(bd), _c(wp), _c(dY)
    cabi.call("npf_resblock1d_bwd", dYc.data_ptr(), xc.data_ptr(), wdc.data_ptr(), bdc.data_ptr(), wpc.data_ptr(), dX.data_ptr(),
              dWd.data_ptr(), dbd.data_ptr() if with_bias_grads else None, dWp.data_ptr(), dbp.data_ptr() if with_bias_grads else None,
              B, L, C, k, PREC["bf16x3"], _st())
    torch.cuda.synchronize()
    assert torch.isfinite(dX).all()
    err = lambda a, b: (a.double().cpu() - b).abs().max().item() / b.abs().max().item()
    checks = [("x", dX, r[0].grad), ("w_dw", dWd - _c(acc0[0]), r[1].grad.view(C, k)), ("w_pw", dWp - _c(acc0[2]), r[3].grad)]
    if with_bias_grads:
        checks += [("b_dw", dbd - _c(acc0[1]), r[2].grad), ("b_pw", dbp - _c(acc0[3]), r[4].grad)]
    else:
        assert torch.equal(dbd, _c(acc0[1])) and torch.equal(dbp, _c(acc0[3]))
    for n, a, b in checks:
        assert err(a, b) < RB_GTOL, (n, err(a, b))
