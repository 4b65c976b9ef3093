"""-m gpu: `bench.py --dump-outputs DIR` writes what the last timed step returned -- the loss and every parameter's gradient --
and those equal a plain eager forward + loss + backward of the same seeded model on that step's seeded inputs; the JSON line
reports the number of steps the timed loop ran.  The comparison runs the project's own kernels (eagerly instead of through the
graph replay), so it pins which step was dumped, the file names, shapes and dtype, not numerical accuracy: the parity tests
against the oracle and the golden vectors cover that."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from _util import ROOT, rel_err

pytestmark = pytest.mark.gpu


def test_dump_outputs_are_the_last_timed_step(tmp_path):
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    steps = 3
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1", "--no-others",
                          "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == steps

    import bench
    import npf_b200
    wl = bench.WORKLOADS["convcnp1d_b256_c128_t128"]
    npf_b200.set_precision("bf16x3")                     # bench.py's default precision
    try:
        model = bench.make_model(wl["family"]).cuda().train()
        inp = bench.make_inputs(wl, wl["B"], seed=(steps - 1) % 4, device="cuda")     # step i replays input set i % 4
        loss = bench.make_loss(wl["loss"]).train()(model(inp["X_cntxt"], inp["Y_cntxt"], inp["X_trgt"], inp["Y_trgt"]), inp["Y_trgt"])
        loss.backward()
        torch.cuda.synchronize()
    finally:
        npf_b200.set_precision("fp32")

    params = dict(model.named_parameters())
    assert sorted(os.listdir(tmp_path)) == sorted(["loss.npy"] + [f"grad.{n}.npy" for n in params])
    got = np.load(tmp_path / "loss.npy")
    assert got.dtype == np.float32 and got.shape == () and rel_err(torch.from_numpy(got), loss) < 1e-5
    for n, p in params.items():
        g = np.load(tmp_path / f"grad.{n}.npy")
        assert g.dtype == np.float32 and g.shape == tuple(p.shape), n
        assert rel_err(torch.from_numpy(g), p.grad) < 1e-3, n
