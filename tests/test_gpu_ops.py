"""-m gpu: every C-ABI kernel family against a plain fp64 torch restatement of the same op (tolerance 1e-4 rel, fp32
path), on shapes that exercise tails, windows and edge cases.  Called through the same ctypes boundary the models use."""
import math

import pytest
import torch
import torch.nn.functional as F

from _util import keep_ids, rel_err

pytestmark = pytest.mark.gpu
TOL = 1e-4   # forward values
GTOL = 1e-3  # gradients (fp32 split reductions / atomics; scalar grads such as d(theta) sum ~1e5 cancelling terms)
# Gradient bars (max-rel) of SetConv and the fused residual block, about 4x the worst error measured on a B200, rounded up.
# The SetConv values gradient runs the split-bf16 tcgen05 kernel in every mode once C = 128 (worst 1.1e-5); the resizer's
# gradients follow the mode.  fp32: 4.5e-5 (few-channel context path); bf16x3: 9e-6 (SetConv), 6.5e-6 (residual block);
# bf16: 2.4e-3.  A split-bf16 product that lost one correction term errs by ~2e-3.
TC_GTOL = {"fp32": 2e-4, "bf16x3": 5e-5, "bf16": 1e-2}


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    import npf_b200
    npf_b200.set_precision("fp32")
    return npf_b200.ops


def _g(*shape, seed=0, scale=1.0):
    return (torch.randn(*shape, generator=torch.Generator().manual_seed(seed), dtype=torch.float64) * scale)


def _cu(t, grad=False):
    return t.float().cuda().requires_grad_(grad)


def _check_grads(cuda_inputs, ref_inputs, out_c, out_r, names, seed=99, gtol=GTOL, scalar_gtol=None):
    """Gradients against fp64 with the bar `gtol`; `scalar_gtol` maps the names of scalar gradients (sums of ~1e5
    cancelling terms, where the bar is relative to a result far below the terms) to their own bar."""
    go = _g(*out_r.shape, seed=seed)
    out_r.backward(go)
    out_c.backward(go.float().cuda())
    for n, c, r in zip(names, cuda_inputs, ref_inputs):
        if r.grad is None:
            continue
        assert c.grad is not None, n
        err = grad_err(c.grad, r.grad)
        bar = (scalar_gtol or {}).get(n, gtol)
        assert err < bar, f"grad {n}: {err} (bar {bar})"


def grad_err(c, r):
    """max |c - r| / max |r|, floored (gradients that are exactly 0 analytically, e.g. dq with one key)."""
    return (c.detach().double().cpu() - r).abs().max().item() / max(r.abs().max().item(), 1e-3)


@pytest.mark.parametrize("M,K,N", [(1, 1, 1), (37, 1, 128), (300, 128, 128), (129, 129, 2), (1000, 3, 32), (513, 256, 130)])
def test_mlp_chain(ops, M, K, N):
    x = _g(M, K, seed=1)
    W1, b1, W2, b2 = _g(N, K, seed=2, scale=K ** -0.5), _g(N, seed=3), _g(7, N, seed=4, scale=N ** -0.5), _g(7, seed=5)
    ref_in = [t.clone().requires_grad_(True) for t in (x, W1, b1, W2, b2)]
    cu_in = [_cu(t, True) for t in (x, W1, b1, W2, b2)]
    yr = F.linear(torch.relu(F.linear(ref_in[0], ref_in[1], ref_in[2])), ref_in[3], ref_in[4])
    yc = ops.mlp_chain(cu_in[0], [cu_in[1], cu_in[3]], [cu_in[2], cu_in[4]])
    assert rel_err(yc, yr) < TOL
    _check_grads(cu_in, ref_in, yc, yr, ["x", "W1", "b1", "W2", "b2"])


@pytest.mark.parametrize("M,K,J", [(5, 1, 1), (1037, 2, 2), (4099, 3, 6), (130, 8, 8), (40000, 2, 2)])
def test_thin_128_layers(ops, M, K, J):
    """x[M,K<=8] -> 128 -> relu -> J<=8: the one-pass thin kernels (forward, fused backward with / without input gradient,
    relu mask taken from the saved activations), rows that do not fill the last warp pass."""
    x = _g(M, K, seed=1)
    W1, b1, W2, b2 = _g(128, K, seed=2, scale=K ** -0.5), _g(128, seed=3), _g(J, 128, seed=4, scale=128 ** -0.5), _g(J, seed=5)
    for x_grad in (True, False):
        ref_in = [t.clone().requires_grad_(True) for t in (x, W1, b1, W2, b2)]
        cu_in = [_cu(t, True) for t in (x, W1, b1, W2, b2)]
        ref_in[0].requires_grad_(x_grad)
        cu_in[0].requires_grad_(x_grad)
        yr = F.linear(torch.relu(F.linear(ref_in[0], ref_in[1], ref_in[2])), ref_in[3], ref_in[4])
        yc = ops.mlp_chain(cu_in[0], [cu_in[1], cu_in[3]], [cu_in[2], cu_in[4]])
        assert rel_err(yc, yr) < TOL
        _check_grads(cu_in, ref_in, yc, yr, ["x", "W1", "b1", "W2", "b2"])
        assert (cu_in[0].grad is not None) == x_grad


def test_linear_final_relu_no_bias(ops):
    x, W = _g(4, 50, 96, seed=1), _g(64, 96, seed=2, scale=0.1)
    xr, Wr = x.clone().requires_grad_(True), W.clone().requires_grad_(True)
    xc, Wc = _cu(x, True), _cu(W, True)
    yr = torch.relu(F.linear(xr, Wr))
    yc = ops.linear(xc, Wc, None, relu=True)
    assert yc.shape == (4, 50, 64) and rel_err(yc, yr) < TOL
    _check_grads([xc, Wc], [xr, Wr], yc, yr, ["x", "W"])


def _setconv_ref(keys, queries, values, theta, W, b):
    k, q, v = keys.unsqueeze(1), queries.unsqueeze(2), values.unsqueeze(1)
    dist = (k - q).abs()
    sigma = 1e-5 + F.softplus(theta)
    a = -(dist / sigma) ** 2
    w = torch.softmax(a, dim=-2)
    dens = torch.exp(a).sum(-2)
    feat = (w * v).sum(2)
    return F.linear(torch.cat([feat, dens], -1), W, b)


@pytest.mark.parametrize("B,K,Q,C,N,regular,sigma,prec", keep_ids([
    (3, 17, 29, 1, 128, False, 0.05, "fp32"),     # context -> induced, tiny
    (2, 128, 384, 2, 128, False, 0.012, "fp32"),  # context -> induced, y_dim 2
    (2, 384, 128, 128, 128, True, 0.012, "fp32"),  # induced -> target at the default length scale (window ~ 20 keys)
    (2, 384, 50, 128, 128, True, 0.2, "fp32"),    # large length scale: window covers most of the grid
    (1, 192, 33, 64, 96, True, 5.0, "fp32"),      # sigma >> grid: dense fallback inside the window code
    (2, 640, 40, 128, 128, True, 0.012, "fp32"),  # extrapolation grid, queries outside [-1, 1]
    (1, 1, 5, 3, 8, False, 0.1, "fp32"),          # single key
    (3, 296, 128, 128, 128, True, 0.012, "fp32"),  # task-resident path (V in shared memory via TMA bulk copies), bench geometry
    (2, 296, 40, 128, 128, True, 0.2, "fp32"),    # task-resident, windows spanning several 32-row chunks
    (149, 296, 9, 128, 128, True, 0.012, "fp32"),  # more tasks than SMs: the persistent CTA loop re-arms its barriers
    (160, 384, 128, 128, 128, True, 0.012, "fp32"),  # bench geometry, 480 key tiles over 148 CTAs: tcgen05 backward, dF restaged per task
    (5, 500, 100, 128, 128, True, 0.03, "fp32"),   # 4 key tiles with a 116-row tail, 2 query chunks with a 36-query tail
    # resizer on tensor cores.  [B*Q, 128] rows: warp-specialised forward with the rank-1 density column (W has 129 columns:
    # scalar weight loads), fused backward accumulating into the 129-column dW
    (3, 296, 128, 128, 128, True, 0.012, "bf16x3"), (3, 296, 128, 128, 128, True, 0.012, "bf16"),
    # 50 rows, fewer than one 128-row tile: separate weight- and data-gradient kernels
    (1, 384, 50, 128, 128, True, 0.2, "fp32"), (1, 384, 50, 128, 128, True, 0.2, "bf16x3"), (1, 384, 50, 128, 128, True, 0.2, "bf16"),
    # 64 channels: the generic tensor-core kernel with the density column, 65-column W / dW
    (2, 384, 100, 64, 128, True, 0.03, "fp32"), (2, 384, 100, 64, 128, True, 0.03, "bf16x3"), (2, 384, 100, 64, 128, True, 0.03, "bf16"),
], "fp32"))
def test_setconv(ops, B, K, Q, C, N, regular, sigma, prec):
    import npf_b200
    npf_b200.set_precision(prec)
    try:
        _run_setconv(ops, B, K, Q, C, N, regular, sigma, prec)
    finally:
        npf_b200.set_precision("fp32")


def _run_setconv(ops, B, K, Q, C, N, regular, sigma, prec):
    gen = torch.Generator().manual_seed(K * 7 + Q)
    if regular:
        grid = torch.linspace(-1.5, 1.5, K).double() if K != 640 else torch.linspace(-2.5, 2.5, K).double()
        keys_r = grid.view(1, K, 1).expand(B, K, 1)
        keys_c = grid.float().cuda()
        span = 2.6 if K == 640 else 1.0
        queries = (torch.rand(B, Q, 1, generator=gen, dtype=torch.float64) * 2 - 1) * span
    else:
        keys_r = torch.rand(B, K, 1, generator=gen, dtype=torch.float64) * 2 - 1
        keys_c = keys_r.float().cuda()
        queries = torch.linspace(-1.5, 1.5, Q).double().view(1, Q, 1).expand(B, Q, 1).contiguous()
    values = _g(B, K, C, seed=3)
    theta = torch.tensor([math.log(math.expm1(sigma))], dtype=torch.float64)
    W, b = _g(N, C + 1, seed=4, scale=(C + 1) ** -0.5), _g(N, seed=5)
    ref_in = [t.clone().requires_grad_(True) for t in (values, theta, W, b)]
    cu_in = [_cu(t, True) for t in (values, theta, W, b)]
    yr = _setconv_ref(keys_r, queries, *ref_in)
    q_c = queries.float().cuda() if regular else queries[0, :, 0].float().cuda()
    yc = ops.setconv(keys_c, q_c, cu_in[0], cu_in[1], cu_in[2], cu_in[3], keys_regular=regular)
    assert rel_err(yc, yr) < (1e-2 if prec == "bf16" else TOL), rel_err(yc, yr)
    _check_grads(cu_in, ref_in, yc, yr, ["values", "theta", "W", "b"], gtol=TC_GTOL[prec], scalar_gtol={"theta": max(GTOL, TC_GTOL[prec])})


@pytest.mark.parametrize("B,K,Q,C,sigma,mode", [
    (3, 128, 384, 1, 0.012, "dup"),       # duplicated context positions, queries sitting exactly on keys
    (2, 700, 257, 3, 0.012, "rand"),      # K > block size: strided sort, y_dim 3
    (2, 40, 384, 1, 0.012, "cluster"),    # all keys clustered far from most queries: windows of the far queries hold every key
    (260, 128, 384, 1, 0.012, "rand"),    # config-2 geometry, more tasks than SMs
    (2, 128, 384, 2, 3.0, "rand"),        # sigma >> key spacing: the window is the whole key set
])
def test_setconv_sorted_small(ops, B, K, Q, C, sigma, mode):
    """The sorted-key few-channel kernel (context -> induced) in the interleaved [feat | dens] layout the model uses
    (values without gradient), against the dense fp64 formula."""
    gen = torch.Generator().manual_seed(K * 3 + Q + C)
    keys_r = torch.rand(B, K, 1, generator=gen, dtype=torch.float64) * 2 - 1
    if mode == "dup":
        keys_r[:, 1::2] = keys_r[:, 0::2]
    if mode == "cluster":
        keys_r = keys_r * 0.01 + 0.8
    grid = torch.linspace(-1.5, 1.5, Q).double()
    if mode == "dup":
        grid[5], grid[100] = keys_r[0, 0, 0], keys_r[0, 2, 0]
    queries = grid.view(1, Q, 1).expand(B, Q, 1).contiguous()
    values = _g(B, K, C, seed=3)
    theta = torch.tensor([math.log(math.expm1(sigma))], dtype=torch.float64)
    N = 128
    W, b = _g(N, C + 1, seed=4, scale=(C + 1) ** -0.5), _g(N, seed=5)
    ref_in = [theta.clone().requires_grad_(True), W.clone().requires_grad_(True), b.clone().requires_grad_(True)]
    cu_in = [_cu(t, True) for t in (theta, W, b)]
    yr = _setconv_ref(keys_r, queries, values, *ref_in)
    yc = ops.setconv(keys_r.float().cuda(), grid.float().cuda(), values.float().cuda(), *cu_in, keys_regular=False)
    assert rel_err(yc, yr) < TOL, rel_err(yc, yr)
    _check_grads(cu_in, ref_in, yc, yr, ["theta", "W", "b"], gtol=TC_GTOL["fp32"], scalar_gtol={"theta": GTOL})


def _dw_ref(x, W, b, res, relu_in, scale, shift):
    nd = x.dim()
    xs = x
    if relu_in:
        if scale is not None:
            xs = xs * scale + shift
        xs = torch.relu(xs)
    xc = xs.permute(0, nd - 1, *range(1, nd - 1))
    C = xc.shape[1]
    pad = W.shape[-1] // 2
    y = F.conv1d(xc, W, b, padding=pad, groups=C) if nd == 3 else F.conv2d(xc, W, b, padding=pad, groups=C)
    y = y.permute(0, *range(2, nd), 1)
    return y + res if res is not None else y


@pytest.mark.parametrize("B,L", [(2, 384), (3, 100), (1, 7), (2, 128), (1, 129), (52, 384), (3, 1000)])
def test_resblock1d_fused(ops, B, L):
    """npf_resblock1d_fwd (depthwise 11 taps + residual + pointwise in one kernel, raw rows by TMA) against the fp64 composite:
    task edges (zero padding inside the halo), row tails, one and several tiles per task, more tiles than CTAs; gradients
    through the autograd Function."""
    import npf_b200
    npf_b200.set_precision("bf16x3")
    try:
        x = _g(B, L, 128, seed=1)
        wd, bd = _g(128, 1, 11, seed=2, scale=0.3), _g(128, seed=3)
        wp, bp = _g(128, 128, 1, seed=4, scale=128 ** -0.5), _g(128, seed=5)
        ref_in = [t.clone().requires_grad_(True) for t in (x, wd, bd, wp, bp)]
        cu_in = [_cu(t, True) for t in (x, wd, bd, wp, bp)]
        xr = ref_in[0]
        o = F.conv1d(torch.relu(xr).transpose(1, 2), ref_in[1], ref_in[2], padding=5, groups=128).transpose(1, 2) + xr
        yr = o @ ref_in[3].view(128, 128).t() + ref_in[4]
        assert ops.resblock1d_supported(cu_in[0], cu_in[1], cu_in[3])
        yc = ops.resblock1d(*cu_in)
        assert torch.isfinite(yc).all()
        assert rel_err(yc, yr) < TOL, rel_err(yc, yr)
        _check_grads(cu_in, ref_in, yc, yr, ["x", "w_dw", "b_dw", "w_pw", "b_pw"], gtol=TC_GTOL["bf16x3"])
    finally:
        npf_b200.set_precision("fp32")


@pytest.mark.parametrize("shape,k,relu_in,affine,res", [
    ((2, 384, 128), 11, True, False, True),
    ((3, 100, 128), 19, True, True, True),
    ((2, 70, 64), 5, False, False, False),
    ((1, 7, 8), 3, True, False, False),
    ((2, 32, 32, 128), 11, True, False, True),
    ((2, 20, 28, 128), 9, True, True, True),
    ((1, 9, 13, 32), 5, False, False, False),
])
def test_dwconv(ops, shape, k, relu_in, affine, res):
    C = shape[-1]
    x = _g(*shape, seed=1)
    W = _g(C, 1, *([k] * (len(shape) - 2)), seed=2, scale=0.3)
    b = _g(C, seed=3)
    r = _g(*shape, seed=4) if res else None
    sc = (_g(C, seed=5).abs() + 0.5) if affine else None
    sh = _g(C, seed=6) if affine else None
    tens = [x, W, b] + ([r] if res else []) + ([sc, sh] if affine else [])
    names = ["x", "W", "b"] + (["res"] if res else []) + (["scale", "shift"] if affine else [])
    ref_in = [t.clone().requires_grad_(True) for t in tens]
    cu_in = [_cu(t, True) for t in tens]

    def unpack(lst):
        it = iter(lst)
        x_, W_, b_ = next(it), next(it), next(it)
        r_ = next(it) if res else None
        sc_, sh_ = (next(it), next(it)) if affine else (None, None)
        return x_, W_, b_, r_, sc_, sh_

    xr, Wr, br, rr, scr, shr = unpack(ref_in)
    xc, Wc, bc, rc, scc, shc = unpack(cu_in)
    yr = _dw_ref(xr, Wr, br, rr, relu_in, scr, shr)
    yc = ops.dwconv(xc, Wc, bc, rc, relu_in, scc, shc)
    assert rel_err(yc, yr) < TOL, rel_err(yc, yr)
    _check_grads(cu_in, ref_in, yc, yr, names)


def test_channel_moments(ops):
    x = _g(5, 77, 128, seed=1) * 3 + 10
    xr, xc = x.clone().requires_grad_(True), _cu(x, True)
    mr, vr = xr.reshape(-1, 128).mean(0), xr.reshape(-1, 128).var(0, unbiased=False)
    mc, vc = ops.channel_moments(xc)
    assert rel_err(mc, mr) < TOL and rel_err(vc, vr) < TOL
    g1, g2 = _g(128, seed=2), _g(128, seed=3)
    (mr * g1 + vr * g2).sum().backward()
    (mc * g1.float().cuda() + vc * g2.float().cuda()).sum().backward()
    assert rel_err(xc.grad, xr.grad) < TOL


@pytest.mark.parametrize("Z,B,T,C,x2_t", [(1, 3, 17, 128, True), (1, 4, 9, 128, False), (5, 2, 11, 64, False), (3, 2, 6, 32, True)])
def test_merge_relu(ops, Z, B, T, C, x2_t):
    x1, x2 = _g(B, T, C, seed=1), _g(Z, B, T if x2_t else 1, C, seed=2)
    r = [t.clone().requires_grad_(True) for t in (x1, x2)]
    c = [_cu(t, True) for t in (x1, x2)]
    yr = torch.relu(r[0].unsqueeze(0) + r[1])
    yc = ops.merge_relu(c[0], c[1])
    assert rel_err(yc, yr) < 1e-6
    _check_grads(c, r, yc, yr, ["x1", "x2"])


def test_mean_pool_layernorm(ops):
    x = _g(6, 13, 128, seed=1)
    xr, xc = x.clone().requires_grad_(True), _cu(x, True)
    yr, yc = xr.mean(1, keepdim=True), ops.mean_pool(xc)
    assert rel_err(yc, yr) < 1e-6
    _check_grads([xc], [xr], yc, yr, ["x"])
    a, b, g, be = _g(7, 19, 128, seed=2), _g(7, 19, 128, seed=3), _g(128, seed=4), _g(128, seed=5)
    r = [t.clone().requires_grad_(True) for t in (a, b, g, be)]
    c = [_cu(t, True) for t in (a, b, g, be)]
    yr = F.layer_norm(r[0] + r[1], (128,), r[2], r[3], 1e-5)
    yc = ops.add_layernorm(*c)
    assert rel_err(yc, yr) < TOL
    _check_grads(c, r, yc, yr, ["a", "b", "gamma", "beta"])


@pytest.mark.parametrize("B,Tq,Tk,H,D,Dv", keep_ids([(2, 33, 70, 8, 16, None), (1, 1, 1, 8, 16, None), (2, 64, 65, 1, 128, None),
                                                      (1, 130, 150, 8, 16, None), (2, 9, 200, 4, 32, None),
                                                      (2, 33, 70, 4, 32, 16)], None))   # Dv None: the value head dim is D
def test_xattn(ops, B, Tq, Tk, H, D, Dv):
    Dv = Dv or D
    q, k, v = _g(B, Tq, H * D, seed=1), _g(B, Tk, H * D, seed=2), _g(B, Tk, H * Dv, seed=3)
    r = [t.clone().requires_grad_(True) for t in (q, k, v)]
    c = [_cu(t, True) for t in (q, k, v)]

    def heads(t, d):
        return t.view(t.shape[0], t.shape[1], H, d).transpose(1, 2)

    s = heads(r[0], D) @ heads(r[1], D).transpose(-1, -2) / math.sqrt(D)
    yr = (s.softmax(-1) @ heads(r[2], Dv)).transpose(1, 2).reshape(B, Tq, H * Dv)
    yc = ops.xattn(c[0], c[1], c[2], H, 1.0 / math.sqrt(D))
    assert yc.shape == yr.shape and rel_err(yc, yr) < TOL, rel_err(yc, yr)
    _check_grads(c, r, yc, yr, ["q", "k", "v"])


def test_gauss_head_and_loglik(ops):
    suff = _g(3, 4, 17, 6, seed=1) * 3
    sr, sc = suff.clone().requires_grad_(True), _cu(suff, True)
    loc_r, s_r = sr.split(3, -1)
    scale_r = 0.01 + 0.99 * F.softplus(s_r)
    loc_c, scale_c = ops.gauss_head(sc, 0.01)
    assert rel_err(loc_c, loc_r) < 1e-6 and rel_err(scale_c, scale_r) < 1e-5
    Y = _g(4, 17, 3, seed=2)
    lp_r = torch.distributions.Normal(loc_r, scale_r).log_prob(Y).reshape(3, 4, -1).sum(-1)
    lp_c = ops.gauss_sum_log_prob(loc_c, scale_c, Y.float().cuda())
    assert rel_err(lp_c, lp_r) < TOL
    _check_grads([sc], [sr], lp_c, lp_r, ["suff"])


def test_latent_sample_global(ops):
    suff, eps = _g(2, 30, 256, seed=1), _g(5, 2, 30, 128, seed=2)
    sr, sc = suff.clone().requires_grad_(True), _cu(suff, True)
    lo_r, s_r = sr.split(128, -1)
    qs_r = 0.1 + 0.9 * torch.sigmoid(s_r)
    z_r = lo_r + qs_r * eps
    lo_c, qs_c, z_c = ops.latent_sample(sc, eps.float().cuda())
    assert rel_err(lo_c, lo_r) < 1e-6 and rel_err(qs_c, qs_r) < 1e-5 and rel_err(z_c, z_r) < 1e-5
    out_r = z_r.sum(0) * 0.3 + lo_r * 0.5 + qs_r * 2.0
    out_c = z_c.sum(0) * 0.3 + lo_c * 0.5 + qs_c * 2.0
    _check_grads([sc], [sr], out_c, out_r, ["suff"])
    z = _g(6, 4, 5, 128, seed=3)
    zr, zc = z.clone().requires_grad_(True), _cu(z, True)
    g_r = torch.cat([zr[..., :64], zr[..., 64:].reshape(6, -1, 64).mean(1).view(6, 1, 1, 64).expand(6, 4, 5, 64)], -1)
    g_c = ops.global_latent(zc)
    assert rel_err(g_c, g_r) < 1e-5
    _check_grads([zc], [zr], g_c, g_r, ["z"])


@pytest.mark.parametrize("B,H,W,y,frac", [(2, 32, 32, 3, 0.3), (1, 20, 28, 1, 0.02), (2, 8, 8, 2, 1.0)])
def test_gridconv_in(ops, B, H, W, y, frac):
    gen = torch.Generator().manual_seed(5)
    img = torch.rand(B, H, W, y, generator=gen, dtype=torch.float64)
    mask = torch.rand(B, H, W, 1, generator=gen) < frac
    Wt = _g(y, 1, 11, 11, seed=2, scale=0.2)
    Wr, Wc = Wt.clone().requires_grad_(True), _cu(Wt, True)
    X = img.permute(0, 3, 1, 2)
    m = mask.permute(0, 3, 1, 2).double()
    sig = F.conv2d(X * m, Wr.abs(), None, padding=5, groups=y)
    den = F.conv2d(m.expand_as(X), Wr.abs(), None, padding=5, groups=y)
    fr = torch.cat([sig / den.clamp(min=1e-5), den], 1).permute(0, 2, 3, 1)
    fc = ops.gridconv_in(img.float().cuda(), mask.cuda(), Wc)
    assert rel_err(fc, fr) < TOL
    _check_grads([Wc], [Wr], fc, fr, ["W"])


def test_range_flag(ops):
    flag = torch.zeros(1, dtype=torch.int32, device="cuda")
    ops.range_flag(flag, torch.rand(1000, device="cuda") * 2 - 1)
    assert int(flag.item()) == 0
    bad = torch.zeros(5000, device="cuda")
    bad[4321] = 1.0001
    ops.range_flag(flag, bad)
    assert int(flag.item()) == 1
    flag.zero_()
    ops.range_flag(flag, torch.tensor([float("nan")], device="cuda"))
    assert int(flag.item()) == 1


def test_cpu_tensors_raise(ops):
    with pytest.raises(RuntimeError):
        ops.linear(torch.randn(3, 4), torch.randn(5, 4))


def test_dwconv_residual_is_input(ops):
    """ResConvBlock with one conv layer: the residual IS the conv input; its gradient is folded into the dX kernel."""
    x, W, b = _g(2, 50, 128, seed=1), _g(128, 1, 11, seed=2, scale=0.3), _g(128, seed=3)
    r = [t.clone().requires_grad_(True) for t in (x, W, b)]
    c = [_cu(t, True) for t in (x, W, b)]
    yr = _dw_ref(r[0], r[1], r[2], r[0], True, None, None)
    yc = ops.dwconv(c[0], c[1], c[2], c[0], True, None, None)
    assert rel_err(yc, yr) < TOL
    _check_grads(c, r, yc, yr, ["x", "W", "b"])
    x2 = _g(1, 5, 6, 32, seed=4)
    W2 = _g(32, 1, 3, 3, seed=5, scale=0.3)
    r2 = [t.clone().requires_grad_(True) for t in (x2, W2)]
    c2 = [_cu(t, True) for t in (x2, W2)]
    yr2 = _dw_ref(r2[0], r2[1], None, r2[0], True, None, None)
    yc2 = ops.dwconv(c2[0], c2[1], None, c2[0], True, None, None)
    assert rel_err(yc2, yr2) < TOL
    _check_grads(c2, r2, yc2, yr2, ["x", "W"])
