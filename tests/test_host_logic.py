"""CPU-only (-m "not gpu") checks of the host side: the C-ABI library loads and exports exactly what include/npf_b200.h
declares, the module trees keep the reference's state_dict keys / parameter counts, constructor error behaviour."""
import ctypes
import os
import re
from functools import partial

import pytest
import torch
import torch.nn as nn

from _cfg import build_model
from _util import ROOT, fixture_names, load_fixture

import npf_b200
from npf_b200 import _cabi
from npf_b200.architectures import CNN, MLP, ResConvBlock, SetConv, get_attender, merge_flat_input


def _header_symbols():
    src = open(os.path.join(ROOT, "include", "npf_b200.h")).read()
    return set(re.findall(r"NPF_API\s+[\w\s\*]+?\b(npf_\w+)\s*\(", src))


def test_cabi_exports_every_declared_symbol():
    declared = _header_symbols()
    assert len(declared) >= 30
    assert os.path.exists(_cabi.LIB_PATH), "libnpf_b200.so not built (run `python __graft_entry__.py build`)"
    lib = ctypes.CDLL(_cabi.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in npf_b200.h but not exported"
    bound = set(_cabi.SIGNATURES) | set(_cabi.BOOKKEEPING)
    assert bound == declared, f"ctypes table and header disagree: {bound ^ declared}"
    lib.npf_abi_version.restype = ctypes.c_int
    assert lib.npf_abi_version() == 1


def test_cabi_argument_validation_without_gpu():
    """Entry points validate their arguments before touching CUDA: callable on a CPU box."""
    lib = _cabi.load()
    rc = lib.npf_linear_fwd(None, 1, None, 1, None, None, 1, 4, 4, 4, 0, None, None, 0, 0, None)
    assert rc == _cabi.NPF_EINVAL
    assert b"null pointer" in lib.npf_last_error()
    with pytest.raises(ValueError):
        _cabi.call("npf_mean_pool_fwd", 1, 1, 2, 0, 8, None)  # N == 0


@pytest.mark.parametrize("name", fixture_names())
def test_state_dict_keys_and_param_counts(name):
    fx = load_fixture(name)
    model = build_model(fx["cfg"])
    missing_unexpected = model.load_state_dict(fx["state_dict"], strict=True)
    assert not missing_unexpected.missing_keys and not missing_unexpected.unexpected_keys
    assert sum(p.numel() for p in model.parameters()) == fx["n_params"]
    assert list(model.state_dict().keys()) == list(fx["state_dict"].keys())  # same order as the reference


def test_notebook_param_counts():
    """Exact structural check against the counts printed by the upstream notebooks (BASELINE.md section 1)."""
    R = 128
    counts = {
        "cnp_notebook_pretrained": 252098, "attncnp_transformer_pretrained": 252738,
        "convcnp_notebook_pretrained": 276612, "gridconvcnp_notebook_pretrained": 340721,
        "convlnp_notebook_pretrained": 376068, "gridconvlnp_notebook_pretrained": 487793,
        "cnp_default": 169922, "attncnp_scaledot": 169922, "convcnp_default": 137476, "gridconvcnp_default_y1": 163195,
    }
    for name, n in counts.items():
        model = build_model(load_fixture(name)["cfg"])
        assert sum(p.numel() for p in model.parameters()) == n, name


def test_constructor_errors_match_reference():
    with pytest.raises(ValueError):
        npf_b200.CNP(1, 1, encoded_path="nonsense")
    with pytest.raises(ValueError):
        get_attender("not-an-attention", 128, 128, 128)
    with pytest.raises(AssertionError):
        SetConv(2, 1, 128)  # x_dim != 1, as upstream setcnn.py:226
    with pytest.raises(AssertionError):
        get_attender("multihead", 100, 100, 100, n_heads=8)  # head divisibility, upstream attention.py:442
    with pytest.raises(AssertionError):
        npf_b200.CNPFLoss()((None, None, object(), None), torch.zeros(1))  # q_zCc must be None, upstream losses.py:116
    with pytest.raises(NotImplementedError):
        MLP(4, 4, activation=nn.Tanh())


def test_model_attributes_and_extrapolation_grid():
    m = npf_b200.ConvCNP(1, 1)
    assert (m.x_dim, m.y_dim, m.r_dim, m.n_induced, m.density_induced) == (1, 1, 128, 384, 128)
    assert torch.allclose(m.X_induced, torch.linspace(-1.5, 1.5, 384))
    m.set_extrapolation((-2, 2))
    assert m.n_induced == int(128 * 5) and abs(float(m.X_induced[0]) + 2.5) < 1e-6
    lm = npf_b200.GridConvLNP(1, 3, n_z_samples_train=16)
    assert isinstance(lm, npf_b200.neuralproc.LatentNeuralProcessFamily) and isinstance(lm, npf_b200.GridConvCNP)
    assert lm.n_z_samples_train == 16 and lm.z_dim == 128


def test_no_cpu_fallback():
    m = npf_b200.CNP(1, 1).eval()
    with pytest.raises(RuntimeError):
        m(torch.rand(2, 3, 1), torch.rand(2, 3, 1), torch.rand(2, 4, 1))


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "neural-process-family_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src.replace("no oracle", ""), f"{f} references the oracle"


def test_product_does_not_read_environment():
    # every kernel choice follows from what the code observes (shapes, precision, alignment, capture, world size): a variable
    # that selects a path nobody tests would let an untested kernel run
    pkg = os.path.join(ROOT, "neural-process-family_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".cu", ".cuh", ".py")):
                src = open(os.path.join(dirpath, f)).read()
                assert "getenv" not in src and "environ" not in src, f"{f} reads the environment"


def test_sync_batchnorm_marks_modules_and_graphed_step_refuses():
    import torch.nn as nn
    from functools import partial
    import npf_b200
    from npf_b200.architectures import CNN, ResConvBlock
    from npf_b200.parallel import sync_batchnorm_
    cnn = partial(CNN, ConvBlock=ResConvBlock, Conv=nn.Conv1d, Normalization=nn.BatchNorm1d, n_blocks=2, kernel_size=5,
                  is_chan_last=True, n_conv_layers=2)
    m = npf_b200.ConvCNP(1, 1, CNN=cnn)
    assert not any(hasattr(b, "_npf_sync_group") for b in m.modules())
    sync_batchnorm_(m)
    bns = [b for b in m.modules() if isinstance(b, nn.BatchNorm1d)]
    assert len(bns) == 4 and all(b._npf_sync_group == (None,) for b in bns)
    with pytest.raises(NotImplementedError):
        npf_b200.GraphedStep(m, npf_b200.CNPFLoss())


def test_checkpoint_roundtrip_and_torch_adam_interchange(tmp_path):
    """Upstream's checkpoint layout (params.pt / optimizer.pt / history.json / eval.csv): save -> load reproduces model,
    moments, step and lr; the optimizer file is a torch.optim.Adam state dict in both directions, including the legacy
    id-keyed layout of upstream's own files."""
    import copy
    import numpy as np
    from npf_b200.parallel import FlatAdam, FlatGradients
    from npf_b200.utils.checkpoint import load_checkpoint, save_checkpoint
    torch.manual_seed(0)
    net = torch.nn.Sequential(torch.nn.Linear(5, 7), torch.nn.ReLU(), torch.nn.Linear(7, 2))
    ref = copy.deepcopy(net)
    ropt = torch.optim.Adam(ref.parameters(), lr=3e-3, betas=(0.8, 0.95), eps=1e-7, weight_decay=0.01)
    for _ in range(3):
        ropt.zero_grad()
        ref(torch.randn(4, 5)).square().sum().backward()
        ropt.step()
    opt = FlatAdam(FlatGradients(net), lr=1.0)
    net.load_state_dict(ref.state_dict())
    opt.load_torch_state_dict(ropt.state_dict())                       # torch -> flat
    assert opt.step_count == 3 and opt.lr == 3e-3 and opt.betas == (0.8, 0.95) and opt.eps == 1e-7 and opt.weight_decay == 0.01
    save_checkpoint(tmp_path, net, opt, history=[dict(epoch=1, train_loss=0.5)], eval_loglik=torch.tensor([1.5, -2.25]))
    assert sorted(os.listdir(tmp_path)) == ["eval.csv", "history.json", "model_summary.txt", "optimizer.pt", "params.pt"]
    assert np.allclose(np.loadtxt(os.path.join(tmp_path, "eval.csv")), [1.5, -2.25])
    net2 = torch.nn.Sequential(torch.nn.Linear(5, 7), torch.nn.ReLU(), torch.nn.Linear(7, 2))
    opt2 = FlatAdam(FlatGradients(net2), lr=9.0)
    hist = load_checkpoint(tmp_path, net2, opt2)
    assert hist == [dict(epoch=1, train_loss=0.5)] and opt2.step_count == 3 and opt2.lr == 3e-3
    assert torch.equal(opt2.exp_avg, opt.exp_avg) and torch.equal(opt2.exp_avg_sq, opt.exp_avg_sq)
    assert all(torch.equal(a, b) for a, b in zip(net2.state_dict().values(), ref.state_dict().values()))
    ropt2 = torch.optim.Adam(net2.parameters())
    ropt2.load_state_dict(torch.load(os.path.join(tmp_path, "optimizer.pt"), weights_only=False))   # flat -> torch
    for a, b in zip(ropt2.state_dict()["state"].values(), ropt.state_dict()["state"].values()):
        assert torch.equal(a["exp_avg"], b["exp_avg"]) and torch.equal(a["exp_avg_sq"], b["exp_avg_sq"]) and int(a["step"]) == 3
    legacy = ropt.state_dict()                                          # upstream's files key the state by id(param)
    ids = [1000 + 7 * i for i in range(len(legacy["param_groups"][0]["params"]))]
    legacy = dict(state={ids[i]: v for i, v in legacy["state"].items()}, param_groups=[dict(legacy["param_groups"][0], params=ids)])
    opt3 = FlatAdam(FlatGradients(copy.deepcopy(net)), lr=9.0)
    opt3.load_torch_state_dict(legacy)
    assert torch.equal(opt3.exp_avg, opt.exp_avg) and opt3.step_count == 3
    with pytest.raises(ValueError):
        opt3.load_torch_state_dict(dict(state={}, param_groups=[dict(legacy["param_groups"][0], params=ids[:-1])]))


def test_train_models_signature_layout_and_eval_csv(tmp_path):
    """npf_b200.utils.train.train_models / eval_loglike (upstream utils/train.py:34-305, utils/evaluate.py:9-28) on the CPU
    with a toy module: loop nest, checkpoint directory layout, best-epoch reload, lr decay, eval.csv in dataset order,
    load-only mode reproducing the stored evaluation."""
    import json
    import numpy as np
    import torch.nn as nn
    from torch.utils.data import TensorDataset
    from npf_b200.utils.train import eval_loglike, train_models

    class Toy(nn.Module):
        def __init__(self):
            super().__init__()
            self.lin = nn.Linear(1, 1)

        def forward(self, X_cntxt, Y_cntxt, X_trgt, Y_trgt=None):
            return (self.lin(X_trgt) + Y_cntxt.mean(1, keepdim=True), None, None, None)

    class ToyLoss(nn.Module):
        def __init__(self, reduction="mean"):
            super().__init__()
            self.reduction = reduction

        def forward(self, pred, Y):
            per_task = ((pred[0] - Y) ** 2).sum((1, 2))
            return per_task if self.reduction is None else per_task.mean(0)

    g = torch.Generator().manual_seed(0)
    x = torch.rand(40, 8, 1, generator=g) * 2 - 1
    y = 3 * x + 0.5
    train, test = TensorDataset(x[:32], y[:32]), TensorDataset(x[32:], y[32:])

    def collate(batch):
        X, Y = torch.stack([b[0] for b in batch]), torch.stack([b[1] for b in batch])
        return dict(X_cntxt=X[:, :3], Y_cntxt=Y[:, :3], X_trgt=X[:, 3:], Y_trgt=Y[:, 3:]), Y[:, 3:]

    kw = dict(criterion=ToyLoss, chckpnt_dirname=str(tmp_path) + "/", device="cpu", max_epochs=6, batch_size=8, lr=5e-2, decay_lr=10, seed=123,
              test_datasets={"toy": test}, train_split=0.25, iterator_train__collate_fn=collate, iterator_valid__collate_fn=collate)
    trainers = train_models({"toy": train}, {"M": Toy}, is_retrain=True, runs=2, **kw)
    assert set(trainers) == {"toy/M/run_0", "toy/M/run_1"}
    t0 = trainers["toy/M/run_0"]
    run_dir = tmp_path / "toy" / "M" / "run_0"
    assert {"params.pt", "optimizer.pt", "history.json", "eval.csv", "model_summary.txt"} <= {p.name for p in run_dir.iterdir()}
    hist = json.load(open(run_dir / "history.json"))
    assert len(hist) == 6 and hist[-1]["train_loss"] < hist[0]["train_loss"]
    assert abs(hist[-1]["lr"] / hist[0]["lr"] - 10 ** (-5 / 6)) < 1e-6               # exponential decay by a total factor 10 over 6 epochs
    assert any(r["valid_loss_best"] for r in hist) and next(p for p in t0.module_.parameters()).device.type == "cpu"
    ev = np.loadtxt(run_dir / "eval.csv", delimiter=",")
    assert ev.shape == (8,)
    ll = eval_loglike(t0, test)                                                        # same numbers, dataset order
    assert np.allclose(ll, ev, rtol=1e-5, atol=1e-6)
    # load-only mode: the stored best checkpoint and eval.csv are returned without training
    loaded = train_models({"toy": train}, {"M": Toy}, is_retrain=False, runs=1, **kw)["toy/M/run_0"]
    for a, b in zip(loaded.module_.parameters(), t0.module_.parameters()):
        assert torch.equal(a, b)
    assert len(loaded.history) == 6
    with pytest.raises(FileNotFoundError):
        train_models({"toy": train}, {"Other": Toy}, is_retrain=False, **kw)


def test_circular_padding_host_logic(monkeypatch):
    """`make_padded_conv(Conv, CircularPad2d)` (upstream helpers.py:334-351, 406-414): wrap-around extension -> the zero-padded
    kernel -> crop must equal a wrap-around convolution.  The CUDA kernels are replaced by torch stand-ins (CPU test of the host logic;
    the kernels themselves run the `*_extrap_pretrained` fixtures in the gpu tests)."""
    import torch.nn.functional as F
    from npf_b200 import ops
    from npf_b200.architectures import cnn as cnn_mod
    from npf_b200.utils.helpers import CircularPad2d, conv_padding, make_abs_conv, make_padded_conv

    def to2nd(t):
        return t.permute(0, 3, 1, 2)

    def fake_dwconv(x, w, b, res, relu_in, sc, sh):
        h = x if sc is None else x * sc + sh
        h = torch.relu(h) if relu_in else h
        y = F.conv2d(to2nd(h), w, b, padding=w.shape[-1] // 2, groups=w.shape[0]).permute(0, 2, 3, 1)
        return y + res if res is not None else y

    def fake_gridconv_in(img, mask, w):
        w = w.abs()
        m = to2nd(mask).to(img.dtype).expand(-1, img.shape[-1], -1, -1)
        pad = w.shape[-1] // 2
        sig = F.conv2d(to2nd(img) * m, w, None, padding=pad, groups=w.shape[0])
        den = F.conv2d(m, w, None, padding=pad, groups=w.shape[0])
        return torch.cat([sig / den.clamp(min=1e-5), den], 1).permute(0, 2, 3, 1)

    monkeypatch.setattr(ops, "dwconv", fake_dwconv)
    monkeypatch.setattr(ops, "gridconv_in", fake_gridconv_in)
    monkeypatch.setattr(ops, "linear", lambda x, w, b: F.linear(x, w, b))
    torch.manual_seed(0)
    conv = make_padded_conv(nn.Conv2d, CircularPad2d)(6, 6, 5, padding=2, groups=6)
    assert conv.padding == (0, 0) and conv_padding(conv)[1] == 2 and isinstance(conv.padder, CircularPad2d)
    x, res = torch.randn(2, 7, 9, 6), torch.randn(2, 7, 9, 6)
    sc, sh = torch.rand(6) + 0.5, torch.randn(6)
    got = cnn_mod._depthwise(x, conv, res, sc, sh)
    want = F.conv2d(F.pad(to2nd(torch.relu(x * sc + sh)), (2,) * 4, mode="circular"), conv.weight, conv.bias, groups=6).permute(0, 2, 3, 1) + res
    assert torch.allclose(got, want, atol=1e-5)
    # pointwise convs built through the same factory carry CircularPad2d(0): plain path
    assert conv_padding(make_padded_conv(nn.Conv2d, CircularPad2d)(6, 4, 1))[0] is None
    # Padder=None keeps the zero padding (upstream :339-342)
    assert make_padded_conv(nn.Conv2d, None)(6, 6, 5, padding=2).padding == (2, 2)

    first = lambda y: make_padded_conv(make_abs_conv(nn.Conv2d), CircularPad2d)(y, y, groups=y, kernel_size=11, padding=5, bias=False)
    m = npf_b200.GridConvCNP(1, 2, Conv=first)
    img, mask = torch.rand(2, 12, 14, 2), torch.rand(2, 12, 14, 1) < 0.3
    got = m.cntxt_to_induced(mask, img)
    w = m.conv.weight.abs()
    mm = to2nd(mask).float().expand(-1, 2, -1, -1)
    wrap = lambda t: F.pad(t, (5,) * 4, mode="circular")
    sig, den = F.conv2d(wrap(to2nd(img) * mm), w, groups=2), F.conv2d(wrap(mm), w, groups=2)
    want = F.linear(torch.cat([sig / den.clamp(min=1e-5), den], 1).permute(0, 2, 3, 1), m.resizer.weight, m.resizer.bias)
    assert torch.allclose(got, want, atol=1e-5)
    with pytest.raises(NotImplementedError):   # a padder the kernels cannot reproduce
        npf_b200.architectures.ResConvBlock(4, 4, make_padded_conv(nn.Conv2d, nn.ReflectionPad2d), kernel_size=3)
