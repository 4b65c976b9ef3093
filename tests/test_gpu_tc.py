"""-m gpu: the tcgen05 / TMEM tensor-core path of the linear layers (NPF_PREC_BF16, NPF_PREC_BF16X3) against fp64
torch: the 3-term split-bf16 mode must meet the fp32 bar (1e-4), plain bf16 the 1e-2 bar of the north star.

Gradient bars.  Where every ReLU mask comes from an input the test supplies (so fp32 and fp64 agree on it), the gradient
error is the arithmetic alone and the bar is set from the worst error measured on a B200, about 4x that rounded up:
GBARS (L2) and GMAX (max-rel).  Split-bf16 with all three products errs by ~5e-6 there, with one correction product
lost by ~2e-3 (CPU emulation, tests/test_tc_bars.py), so these bars tell the two apart.  test_tc_mlp_chain computes its
masks from fp32 pre-activations and keeps the looser ReLU-flip bar of BARS."""
import pytest
import torch
import torch.nn.functional as F

from _cfg import build_model, loss_for
from _util import keep_ids, load_fixture, rel_err

pytestmark = pytest.mark.gpu
BARS = {"bf16": (1e-2, 2e-1), "bf16x3": (1e-4, 3e-3)}   # (forward max-rel, gradient L2-rel with ReLU flips) tolerances
# flip-free gradient bars; worst error measured on a B200 (bf16x3 / bf16) in the comment.  The one-layer bar is 5e-5
# rather than 2e-5 so that it stays 5x above the emulated split-bf16 error (4.5e-6; tests/test_tc_bars.py)
GBARS = {"bf16x3": 5e-5, "bf16": 1e-2}          # L2-rel, one layer (npf_linear_bwd): 4.7e-6 / 2.4e-3
CHAIN_GBARS = {"bf16x3": 1e-4, "bf16": 5e-2}    # L2-rel, npf_mlp_chain_bwd (up to 8 layers): 1.3e-5 / 6.7e-3
GMAX = {"bf16x3": 5e-5}                         # max-rel, one layer through npf_b200.ops.linear: 7.9e-6
ABARS = {"bf16x3": 5e-5, "bf16": 2e-2}          # L2-rel, attention: 7.2e-6 / 4.9e-3
ZERO_GRAD_BARS = {"bf16x3": 2e-3, "bf16": 5e-2}  # attention gradients that are 0 analytically: cancellation only, 3.3e-4 / 2.7e-2


def l2_rel(a, b):
    """||a - b||_2 / ||b||_2.  Gradients of ReLU chains are compared in L2: a pre-activation within rounding distance of
    0 flips its mask and moves ONE sample's gradient row by O(1) -- a max-norm metric then measures how many of the ~1e6
    units happen to sit within 1e-5 of zero, not the arithmetic."""
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


def grad_max_rel(a, b):
    """max |a - b| / max |b| of a gradient (rel_err under its own name, so each bar's metric reads at the call)."""
    return rel_err(a, b)


@pytest.fixture(scope="module")
def npf():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    import npf_b200
    yield npf_b200
    npf_b200.set_precision("fp32")


def _g(*shape, seed=0, scale=1.0):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed), dtype=torch.float64) * scale


@pytest.mark.parametrize("prec", ["bf16x3", "bf16"])
@pytest.mark.parametrize("M,K,H,N", [(1, 128, 128, 128), (300, 128, 128, 128), (1000, 64, 128, 32), (4099, 128, 256, 16), (130, 128, 128, 2),
                                     (32768, 128, 128, 128)])
def test_tc_mlp_chain(npf, prec, M, K, H, N):
    npf.set_precision(prec)
    ftol, gtol = BARS[prec]
    ts = [_g(M, K, seed=1), _g(H, K, seed=2, scale=K ** -0.5), _g(H, seed=3), _g(H, H, seed=4, scale=H ** -0.5), _g(H, seed=5),
          _g(N, H, seed=6, scale=H ** -0.5), _g(N, seed=7)]
    r = [t.clone().requires_grad_(True) for t in ts]
    c = [t.float().cuda().requires_grad_(True) for t in ts]
    yr = F.linear(torch.relu(F.linear(torch.relu(F.linear(r[0], r[1], r[2])), r[3], r[4])), r[5], r[6])
    yc = npf.ops.mlp_chain(c[0], [c[1], c[3], c[5]], [c[2], c[4], c[6]])
    assert rel_err(yc, yr) < ftol, rel_err(yc, yr)
    go = _g(*yr.shape, seed=9)
    yr.backward(go)
    yc.backward(go.float().cuda())
    for n, a, b in zip("x W1 b1 W2 b2 W3 b3".split(), c, r):
        err = l2_rel(a.grad, b.grad)
        assert err < gtol, f"{prec} grad {n}: {err}"


@pytest.mark.parametrize("prec", ["bf16x3", "bf16"])
@pytest.mark.parametrize("M,mask,bias", [(128, True, True), (1000, True, True), (4099, False, True), (75776, True, False), (640, False, False)])
def test_tc_fused_linear_backward(npf, prec, M, mask, bias):
    """npf_linear_bwd on the 128 -> 128 hot shape (one pass: dX, dW +=, db +=) against fp64, including row tails, the relu
    mask taken from the staged X tile, accumulation into non-zero dW / db, and agreement with the two-kernel path."""
    from npf_b200 import _cabi
    K = N = 128
    pr = {"bf16": 1, "bf16x3": 2}[prec]
    gtol = GBARS[prec]
    dY, W = _g(M, N, seed=1), _g(N, K, seed=2, scale=K ** -0.5)
    X = torch.relu(_g(M, K, seed=3))
    dW0, db0 = _g(N, K, seed=4), _g(N, seed=5)
    dXr = dY @ W
    if mask:
        dXr = dXr * (X > 0)
    dWr, dbr = dW0 + dY.t() @ X, db0 + dY.sum(0)
    c = lambda t: t.float().cuda().contiguous()
    dYc, Wc, Xc, dWc, dbc = c(dY), c(W), c(X), c(dW0), c(db0)
    dXc = torch.full((M, K), float("nan"), device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    _cabi.call("npf_linear_bwd", dYc.data_ptr(), N, Xc.data_ptr(), K, Wc.data_ptr(), K, dXc.data_ptr(), K, dWc.data_ptr(), K,
               dbc.data_ptr() if bias else 0, M, K, N, 16 if mask else 0, pr, st)
    torch.cuda.synchronize()
    assert torch.isfinite(dXc).all()
    assert l2_rel(dXc, dXr) < gtol, l2_rel(dXc, dXr)
    assert l2_rel(dWc - c(dW0), dWr - dW0) < gtol, l2_rel(dWc - c(dW0), dWr - dW0)
    if bias:
        assert l2_rel(dbc - c(db0), dbr - db0) < gtol
    else:
        assert torch.equal(dbc, c(db0))
    if mask:   # masked entries are exact zeros
        assert (dXc[(Xc <= 0)] == 0).all()
    # the separate kernels give the same numbers to rounding
    dW2, dX2 = c(dW0), torch.empty(M, K, device="cuda")
    _cabi.call("npf_linear_bwd_weight", dYc.data_ptr(), N, Xc.data_ptr(), K, dW2.data_ptr(), K, 0, M, K, N, 0, 0, 0, 0, pr, st)
    _cabi.call("npf_linear_bwd_data", dYc.data_ptr(), N, Wc.data_ptr(), K, dX2.data_ptr(), K, M, K, N, Xc.data_ptr() if mask else 0,
               K if mask else 0, 0, pr, st)
    assert l2_rel(dXc, dX2) < 1e-5 and l2_rel(dWc - c(dW0), dW2 - c(dW0)) < (1e-5 if prec == "bf16x3" else 1e-4)


@pytest.mark.parametrize("prec", ["bf16x3", "bf16"])
@pytest.mark.parametrize("L,M,relu_mask,relu_in", [(2, 1, 0b01, 0), (5, 257, 0b01111, 0), (8, 4099, 0b10110101, 1), (4, 37888, 0b0111, 0), (3, 40000, 0b011, 0), (4, 131072, 0b1111, 0)])
def test_tc_mlp_chain_entry(npf, prec, L, M, relu_mask, relu_in):
    """npf_mlp_chain_fwd (row block kept on chip between layers) against the same layers run one npf_linear_fwd at a time and
    against fp64: every saved activation, missing biases, arbitrary ReLU pattern, partial tiles, and the size fallback."""
    import ctypes
    from npf_b200 import _cabi
    pr = {"bf16": 1, "bf16x3": 2}[prec]
    ftol, _ = BARS[prec]
    st = torch.cuda.current_stream().cuda_stream
    X = _g(M, 128, seed=1)
    Ws = [_g(128, 128, seed=10 + l, scale=128 ** -0.5) for l in range(L)]
    bs = [None if l % 3 == 1 else _g(128, seed=30 + l) for l in range(L)]
    Xc, Wc = X.float().cuda(), [w.float().cuda() for w in Ws]
    bc = [None if b is None else b.float().cuda() for b in bs]
    Ys = [torch.full((M, 128), float("nan"), device="cuda") for _ in range(L)]
    Wp = (ctypes.c_void_p * L)(*[w.data_ptr() for w in Wc])
    bp = (ctypes.c_void_p * L)(*[None if b is None else b.data_ptr() for b in bc])
    Yp = (ctypes.c_void_p * L)(*[y.data_ptr() for y in Ys])
    _cabi.call("npf_mlp_chain_fwd", Xc.data_ptr(), 128, Wp, bp, Yp, L, M, 128, relu_in, relu_mask, pr, st)
    h64 = torch.relu(X) if relu_in else X
    hseq = Xc
    for l in range(L):
        h64 = h64 @ Ws[l].t() + (0 if bs[l] is None else bs[l])
        if (relu_mask >> l) & 1:
            h64 = torch.relu(h64)
        y = torch.empty(M, 128, device="cuda")
        flags = (2 if (l == 0 and relu_in) else 0) | (1 if (relu_mask >> l) & 1 else 0)
        _cabi.call("npf_linear_fwd", hseq.data_ptr(), 128, Wc[l].data_ptr(), 128, 0 if bc[l] is None else bc[l].data_ptr(), y.data_ptr(), 128, M, 128, 128,
                   flags, 0, 0, 0, pr, st)
        hseq = y
        assert torch.isfinite(Ys[l]).all()
        assert rel_err(Ys[l], h64) < ftol * (l + 1), (l, rel_err(Ys[l], h64))
        assert l2_rel(Ys[l], y) < (2e-5 if prec == "bf16x3" else 1e-2) * (l + 1), (l, l2_rel(Ys[l], y))


@pytest.mark.parametrize("prec", ["bf16x3", "bf16"])
@pytest.mark.parametrize("L,M,need_dx,mask0", [(2, 64, True, False), (4, 100, True, True), (5, 257, False, False), (4, 1024, True, False),
                                               (4, 32768, True, False), (3, 40000, True, True), (8, 4099, True, False)])
def test_tc_mlp_chain_bwd_entry(npf, prec, L, M, need_dx, mask0):
    """npf_mlp_chain_bwd (gradient kept on chip between the layers) against fp64: dX, every dW (accumulated into a non-zero
    buffer) and db (one entry NULL), partial 64-row blocks, one and several row groups per CTA, with / without dX and input mask."""
    import ctypes
    from npf_b200 import _cabi
    pr = {"bf16": 1, "bf16x3": 2}[prec]
    gtol = CHAIN_GBARS[prec]
    st = torch.cuda.current_stream().cuda_stream
    Ws = [_g(128, 128, seed=10 + l, scale=128 ** -0.5) for l in range(L)]
    X0 = _g(M, 128, seed=1)
    if mask0:
        X0 = torch.relu(X0)
    Xs = [X0]
    for l in range(L - 1):                                           # saved inputs: post-ReLU outputs of the previous layer
        Xs.append(torch.relu(Xs[-1] @ Ws[l].t() + 0.1 * _g(128, seed=40 + l)))
    dY = _g(M, 128, seed=2)
    dW0 = [_g(128, 128, seed=60 + l) for l in range(L)]
    db0 = [_g(128, seed=80 + l) for l in range(L)]
    # fp64 reference
    dz, dWr, dbr = dY, [None] * L, [None] * L
    for l in range(L - 1, -1, -1):
        dWr[l] = dz.t() @ Xs[l]
        dbr[l] = dz.sum(0)
        dz = dz @ Ws[l]
        if l > 0 or mask0:
            dz = dz * (Xs[l] > 0)
    c = lambda t: t.float().cuda().contiguous()
    Xc, Wc, dWc, dbc, dYc = [c(x) for x in Xs], [c(w) for w in Ws], [c(w) for w in dW0], [c(b) for b in db0], c(dY)
    skip_db = 1 if L > 2 else -1
    dXc = torch.full((M, 128), float("nan"), device="cuda") if need_dx else None
    arr = lambda ts: (ctypes.c_void_p * L)(*[None if t is None else t.data_ptr() for t in ts])
    _cabi.call("npf_mlp_chain_bwd", dYc.data_ptr(), 128, arr(Xc), arr(Wc), None if dXc is None else dXc.data_ptr(), 128, arr(dWc),
               arr([None if l == skip_db else dbc[l] for l in range(L)]), L, M, 128, 16 if mask0 else 0, pr, st)
    torch.cuda.synchronize()
    if need_dx:
        assert torch.isfinite(dXc).all()
        assert l2_rel(dXc, dz) < gtol, ("dX", l2_rel(dXc, dz))
        if mask0:
            assert (dXc[Xc[0] <= 0] == 0).all()
    for l in range(L):
        e = l2_rel(dWc[l] - c(dW0[l]), dWr[l])
        assert e < gtol, (f"dW{l}", e)
        if l == skip_db:
            assert torch.equal(dbc[l], c(db0[l]))
        else:
            e = l2_rel(dbc[l] - c(db0[l]), dbr[l])
            assert e < gtol, (f"db{l}", e)


@pytest.mark.parametrize("prec", ["bf16x3", "bf16"])
def test_tc_model_parity_convcnp(npf, prec):
    """Whole ConvCNP (pointwise convs, SetConv resizer with the rank-1 density column, decoder MLP) on tensor cores."""
    npf.set_precision(prec)
    ftol = {"bf16x3": 1e-4, "bf16": 3e-2}[prec]   # plain bf16 through the 10-GEMM-deep stack: ~2e-2 (DESIGN.md section 4)
    fx = load_fixture("convcnp_default")
    model = build_model(fx["cfg"])
    model.load_state_dict(fx["state_dict"])
    model.cuda().train()
    for case in fx["cases"][:2]:
        model.zero_grad(set_to_none=True)
        inp = {k: v.cuda() for k, v in case["inputs"].items()}
        out = model(inp["X_cntxt"], inp["Y_cntxt"], inp["X_trgt"], inp["Y_trgt"])
        per_task = loss_for("cnpf")(out, inp["Y_trgt"])
        assert rel_err(out[0].base_dist.loc, case["loc"]) < ftol, (prec, rel_err(out[0].base_dist.loc, case["loc"]))
        assert rel_err(out[0].base_dist.scale, case["scale"]) < ftol
        assert rel_err(per_task, case["loss_per_task"]) < ftol


@pytest.mark.parametrize("prec", ["bf16x3"])
@pytest.mark.parametrize("M,K,N", [(513, 128, 128), (513, 128, 256), (513, 16, 256), (513, 64, 32), (513, 128, 16), (70000, 128, 128),
                                   (513, 256, 16), (513, 32, 128)])
def test_tc_single_linear_localised(npf, prec, M, K, N):
    """One layer at a time (forward, data gradient, weight gradient reported separately) + run-to-run determinism of
    the forward and of the data gradient (no atomics on those paths)."""
    npf.set_precision(prec)
    ftol, gtol = BARS[prec][0], GMAX[prec]
    x, W, b = _g(M, K, seed=1), _g(N, K, seed=2, scale=K ** -0.5), _g(N, seed=3)
    go = _g(M, N, seed=4)
    res = []
    for rep in range(2):
        xc, Wc, bc = (t.float().cuda().requires_grad_(True) for t in (x, W, b))
        yc = npf.ops.linear(xc, Wc, bc)
        yc.backward(go.float().cuda())
        res.append((yc.detach().clone(), xc.grad.clone(), Wc.grad.clone(), bc.grad.clone()))
    yr = x @ W.t() + b
    errs = dict(y=rel_err(res[0][0], yr), dx=grad_max_rel(res[0][1], go @ W), dW=grad_max_rel(res[0][2], go.t() @ x),
                db=grad_max_rel(res[0][3], go.sum(0)))
    assert torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][1], res[1][1]), f"non-deterministic: {errs}"
    assert errs["y"] < ftol and errs["dx"] < gtol and errs["dW"] < gtol and errs["db"] < gtol, errs


def attn_grad_err(a, b, gmax, floor):
    """L2 error of one attention gradient relative to its own norm, floored at a fraction of the largest of the three
    (with a single key the softmax gradient w.r.t. q and k is exactly 0: only cancellation is left to compare)."""
    return (a.detach().double().cpu() - b).norm().item() / max(b.norm().item(), floor * gmax)


def attn_ref(q, k, v, H, D, Dv):
    """fp64 softmax attention over H heads; q, k [B, T, H*D], v [B, Tk, H*Dv]."""
    import math
    heads = lambda t, d: t.view(t.shape[0], t.shape[1], H, d).transpose(1, 2)
    s = heads(q, D) @ heads(k, D).transpose(-1, -2) / math.sqrt(D)
    return (s.softmax(-1) @ heads(v, Dv)).transpose(1, 2).reshape(q.shape[0], q.shape[1], H * Dv)


@pytest.mark.parametrize("prec", ["bf16x3", "bf16"])
@pytest.mark.parametrize("B,Tq,Tk,H,D,Dv", keep_ids([
    (2, 128, 128, 8, 16, None), (1, 33, 70, 8, 16, None), (2, 300, 513, 4, 32, None), (1, 1, 1, 8, 16, None), (2, 512, 512, 8, 16, None),
    (38, 128, 100, 8, 16, None),    # 304 CTAs: 64-key chunks, a 36-key tail
    (40, 130, 513, 8, 32, None),    # 64-key chunks with head dim 32, query and key tails
    (2, 33, 70, 8, 16, 32), (1, 130, 150, 8, 32, 16),        # value head dim Dv != query / key head dim D, 128-key chunks
    (40, 130, 100, 4, 16, 32), (40, 130, 100, 4, 32, 16),    # ... and with 64-key chunks (320 CTAs)
], None))   # Dv None: the value head dim is D
def test_tc_attention_forward(npf, prec, B, Tq, Tk, H, D, Dv):
    """tcgen05 attention forward + backward (head dims 16 / 32, also mixed between q/k and v) vs fp64 softmax attention."""
    import math
    Dv = Dv or D
    npf.set_precision(prec)
    ftol = {"bf16x3": 1e-4, "bf16": 1e-2}[prec]
    q, k, v = _g(B, Tq, H * D, seed=1), _g(B, Tk, H * D, seed=2), _g(B, Tk, H * Dv, seed=3)
    r = [t.clone().requires_grad_(True) for t in (q, k, v)]
    yr = attn_ref(*r, H, D, Dv)
    c = [t.float().cuda().requires_grad_(True) for t in (q, k, v)]
    yc = npf.ops.xattn(c[0], c[1], c[2], H, 1.0 / math.sqrt(D))
    assert yc.shape == yr.shape
    assert rel_err(yc, yr) < ftol, (prec, rel_err(yc, yr))
    go = _g(*yr.shape, seed=9)
    yr.backward(go)
    yc.backward(go.float().cuda())
    gmax = max(t_.grad.norm().item() for t_ in r)
    floor = {"bf16x3": 1e-2, "bf16": 5e-2}[prec]
    for n, a, b_ in zip("qkv", c, r):
        err = attn_grad_err(a.grad, b_.grad, gmax, floor)
        # a gradient below the floor is 0 analytically (one key: dq = dk = 0) and what is left is cancellation
        bar = ABARS[prec] if b_.grad.norm().item() >= floor * gmax else ZERO_GRAD_BARS[prec]
        assert err < bar, f"{prec} grad {n}: {err}"


from _util import fixture_names  # noqa: E402


@pytest.mark.parametrize("name", fixture_names())
def test_tc_x3_all_models_match_golden(npf, name):
    """Every model family in the split-bf16 tensor-core mode (linear layers, attention) against the reference's golden
    vectors.  The products of this mode carry ~16 bits (2^-16 ~ 1.5e-5): 1e-4 on mu, sigma, loss holds for every fixture
    except the upstream-pretrained transformer-attention checkpoints (AttnCNP / AttnLNP, cross- and self-attention), whose
    sharp attention / large weights amplify it to 1e-4 .. 3e-4 (bar 5e-4 here; the fp32 mode meets 1e-4 on all of them,
    tests/test_gpu_parity.py; measured per case by profiles/microbench/fixture_errors.py)."""
    tol = 5e-4 if name in ("attncnp_transformer_pretrained", "attncnp_selfattn_pretrained", "attnlnp_pretrained",
                           "attnlnp_selfattn_pretrained") else 1e-4
    npf.set_precision("bf16x3")
    fx = load_fixture(name)
    model = build_model(fx["cfg"])
    model.load_state_dict(fx["state_dict"])
    model.cuda()
    for case in fx["cases"]:
        model.load_state_dict(fx["state_dict"])
        model.train(case["training"])
        if "extrap" in case:
            model.set_extrapolation(tuple(case["extrap"]))
        if "eps" in case:
            model._eps_override = case["eps"].cuda()
        inp = {k: v.cuda() for k, v in case["inputs"].items()}
        crit = loss_for(case["loss_name"])
        crit.train(case["training"])
        out = model(inp["X_cntxt"], inp["Y_cntxt"], inp["X_trgt"], inp["Y_trgt"])
        per_task = crit(out, inp["Y_trgt"])
        tag = f"{name}/{case['name']}"
        # loc is measured against max(|loc|, 1 % of the predictive std): with no context the ConvCNP mean is ~2e-4 while
        # sigma is 0.7 -- the fp32 reference itself only matches its fp64 re-run to 3e-5 of |loc| there
        loc, ref_loc = out[0].base_dist.loc.detach().double().cpu(), case["loc"].double()
        e_loc = ((loc - ref_loc).abs().max() / max(ref_loc.abs().max().item(), 1e-2 * case["scale"].abs().max().item())).item()
        assert e_loc < tol, f"{tag} loc {e_loc}"
        assert rel_err(out[0].base_dist.scale, case["scale"]) < tol, f"{tag} scale {rel_err(out[0].base_dist.scale, case['scale'])}"
        assert rel_err(per_task, case["loss_per_task"]) < tol, f"{tag} loss {rel_err(per_task, case['loss_per_task'])}"
        if "extrap" in case:
            model.set_extrapolation((-1, 1))
