"""Shared helpers for the test-suite: fixture loading, running the CPU oracle on a fixture case,
gradient projections (the compact gradient pin stored in tests/golden/*.pt)."""
import glob
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG_DIR = os.path.join(ROOT, "neural-process-family_b200")
for p in (ROOT, PKG_DIR):
    if p not in sys.path:
        sys.path.insert(0, p)

from oracle import npf_oracle as O  # noqa: E402  (test infrastructure only)

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")
N_PROJ = 8


def fixture_names():
    return sorted(os.path.splitext(os.path.basename(p))[0] for p in glob.glob(os.path.join(GOLDEN_DIR, "*.pt")))


def load_fixture(name):
    fx = torch.load(os.path.join(GOLDEN_DIR, name + ".pt"), map_location="cpu", weights_only=False)
    for case in fx["cases"]:
        if "eps_seed" in case and "eps" not in case:
            # a large eps is stored as (seed, shape, checksum) by oracle/gen_golden.py and regenerated here
            e = torch.randn(tuple(case["eps_shape"]), generator=torch.Generator().manual_seed(case["eps_seed"]))
            chk = torch.stack([e.double().sum(), e.double().abs().sum(), e.reshape(-1)[:: max(1, e.numel() // 7)].double().sum()])
            assert torch.allclose(chk, case["eps_check"], rtol=0, atol=1e-9), f"{name}: eps regenerated from its seed differs from the recorded one"
            case["eps"] = e
    return fx


def grad_projection(g):
    """Same compact pin as oracle/gen_golden.py::grad_projection (8 random projections + L2 norm)."""
    out = []
    g64 = g.detach().double().reshape(-1).cpu()
    for i in range(N_PROJ):
        v = torch.randn(g64.numel(), generator=torch.Generator().manual_seed(1000 + i), dtype=torch.float64)
        out.append(torch.dot(g64, v))
    out.append(g64.norm())
    return torch.stack(out)


def is_param(name):
    return not ("running_" in name or "num_batches_tracked" in name)


def oracle_run(cfg, state_dict, case, dtype=torch.float32, with_grads=False):
    """Run the CPU oracle on one fixture case.  Returns dict(loc, scale, loss_per_task, loss, grads?)."""
    sd = {}
    for k, v in state_dict.items():
        if v.is_floating_point():
            t = v.detach().clone().to(dtype)
            if with_grads and is_param(k):
                t.requires_grad_(True)
            sd[k] = t
        else:
            sd[k] = v.clone()
    inp = case["inputs"]
    cast = lambda t: t.to(dtype) if t.is_floating_point() else t
    Xc, Yc, Xt, Yt = (cast(inp[k]) for k in ("X_cntxt", "Y_cntxt", "X_trgt", "Y_trgt"))
    fam = cfg["family"]
    training = case["training"]
    extra = {}
    if fam == "CNP":
        loc, scale = O.cnp_forward(sd, Xc, Yc, Xt)
    elif fam == "AttnCNP":
        loc, scale = O.attncnp_forward(sd, Xc, Yc, Xt, attention=cfg.get("attention", "scaledot"),
                                       is_self_attn=cfg.get("is_self_attn", False))
    elif fam == "AttnLNP":
        # z ~ q(z | targets) whenever the targets are known and is_q_zCct (base.py:501), train or eval
        loc, scale, z, (q_loc, q_scale), q_ct = O.attnlnp_forward(
            sd, Xc, Yc, Xt, cast(case["eps"]), attention=cfg.get("attention", "scaledot"),
            is_self_attn=cfg.get("is_self_attn", False), Y_trgt=Yt if cfg.get("is_q_zCct") else None)
        extra.update(q_loc=q_loc, q_scale=q_scale)
        if q_ct is not None:
            extra.update(q_ct_loc=q_ct[0], q_ct_scale=q_ct[1])
    elif fam == "ConvCNP":
        Xi = _induced(cfg, case, dtype)
        loc, scale = O.convcnp_forward(sd, Xc, Yc, Xt, X_induced=Xi, training=training)
    elif fam == "GridConvCNP":
        loc, scale = O.gridconvcnp_forward(sd, Xc, Yc, Xt, training=training, **_conv_opts(cfg))
    elif fam == "LNP":
        eps = cast(case["eps"])
        if cfg.get("is_q_zCct") and training:
            # q(z|cntxt,trgt) sampling: base.py:501-506 encodes the targets with the same encoder
            loc, scale, z, q_loc, q_scale, q_ct = _lnp_qzct(sd, Xc, Yc, Xt, Yt, eps, cfg)
            extra.update(q_ct_loc=q_ct[0], q_ct_scale=q_ct[1])
        else:
            loc, scale, z, q_loc, q_scale = O.lnp_forward(sd, Xc, Yc, Xt, eps, cfg.get("encoded_path", "latent"))
        extra.update(q_loc=q_loc, q_scale=q_scale)
    elif fam == "ConvLNP":
        Xi = _induced(cfg, case, dtype)
        loc, scale, z, q_loc, q_scale = O.convlnp_forward(
            sd, Xc, Yc, Xt, cast(case["eps"]), X_induced=Xi, is_global=cfg.get("is_global", False), training=training)
        extra.update(q_loc=q_loc, q_scale=q_scale)
    elif fam == "GridConvLNP":
        loc, scale, z, q_loc, q_scale = O.gridconvlnp_forward(
            sd, Xc, Yc, cast(case["eps"]), is_global=cfg.get("is_global", False), training=training, **_conv_opts(cfg))
        extra.update(q_loc=q_loc, q_scale=q_scale)
    else:
        raise ValueError(fam)

    ln = case["loss_name"]
    if ln == "cnpf":
        per_task = O.cnpf_loss(loc, scale, Yt, reduction=None)
    elif ln == "nll" or not training:
        per_task = O.nll_lnpf_loss(loc, scale, Yt, reduction=None)
    elif ln == "elbo":
        per_task = O.elbo_lnpf_loss(loc, scale, Yt, extra["q_ct_loc"], extra["q_ct_scale"], extra["q_loc"],
                                    extra["q_scale"], reduction=None)
    loss = per_task.mean(0)
    out = dict(loc=loc.detach(), scale=scale.detach(), loss_per_task=per_task.detach(), loss=loss.detach())
    out.update({k: v.detach() for k, v in extra.items()})
    if with_grads:
        loss.backward()
        out["grads"] = {k: v.grad.detach() for k, v in sd.items() if v.is_floating_point() and v.grad is not None}
    return out


def _conv_opts(cfg):
    return dict(circular=bool(cfg.get("circular", False)), bn_eps=cfg.get("cnn", {}).get("bn_eps", 1e-5))


def _induced(cfg, case, dtype):
    if "X_induced" in case:
        return case["X_induced"].to(dtype)
    return O.induced_grid(cfg.get("density_induced", 128)).to(dtype)


def _lnp_qzct(sd, Xc, Yc, Xt, Yt, eps, cfg):
    """LNP with is_q_zCct=True in training (base.py:495-514): z ~ q(z | targets)."""
    Xe_t = O.mlp(sd, "x_encoder.", Xt)
    R_t = O.merge_flat_sum(sd, "xy_encoder.", Xe_t, Yt).mean(dim=1, keepdim=True)
    z_dim = sd["latent_encoder.out.weight"].shape[0] // 2
    suff = O.mlp(sd, "latent_encoder.", R_t)
    q_ct_loc, s = suff.split(z_dim, dim=-1)
    q_ct_scale = O.q_z_scale(s)
    Xe_c = O.mlp(sd, "x_encoder.", Xc)
    R = O.merge_flat_sum(sd, "xy_encoder.", Xe_c, Yc).mean(dim=1, keepdim=True)
    suff_c = O.mlp(sd, "latent_encoder.", R)
    q_loc, s_c = suff_c.split(z_dim, dim=-1)
    q_scale = O.q_z_scale(s_c)
    z = q_ct_loc.unsqueeze(0) + q_ct_scale.unsqueeze(0) * eps
    r_dim = R.shape[-1]
    if cfg.get("encoded_path", "latent") == "both":
        Rz = R.unsqueeze(0).expand(*z.shape[:-1], r_dim)
        R_trgt = torch.relu(torch.nn.functional.linear(torch.cat((Rz, z), -1), sd["r_z_merger.weight"], sd["r_z_merger.bias"]))
    else:
        R_trgt = z
    R_trgt = R_trgt.expand(z.shape[0], Xt.shape[0], Xt.shape[1], r_dim)
    loc, scale = O._decode(sd, Xe_t, R_trgt, Yc.shape[-1])
    return loc, scale, z, q_loc, q_scale, (q_ct_loc, q_ct_scale)


def rel_err(a, b):
    """max |a-b| / max(|b|, tiny): the 'rel' used for the 1e-4 fp32 / 1e-2 bf16 parity bars."""
    a = a.detach().double().cpu()
    b = b.detach().double().cpu()
    if a.numel() == 0:
        return 0.0
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-30)).item()


def keep_ids(cases, default):
    """pytest.params whose id leaves out the last column when it holds `default`: the cases that existed before that
    column was added keep their test ids."""
    return [pytest.param(*c, id="-".join(map(str, c if c[-1] != default else c[:-1]))) for c in cases]
