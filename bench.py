#!/usr/bin/env python
"""bench.py -- tasks/sec of one meta-batch forward + loss + backward (the BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--precision P]
                    [--dump-outputs DIR]

Default workload = BASELINE.json configs[1]: ConvCNP(1,1) default constructor (I=384 induced points, 3 ResConvBlocks
k=11), meta-batch 256 tasks PER GPU, 128 context / 128 target points, fp32 storage, synthetic data (random-init
weights under seed 0, X ~ U(-1,1), Y ~ N(0,1)).  Weak scaling: every rank processes its own 256 tasks; for N > 1 the
flat gradient is all-reduced (NCCL) inside the timed region.  One JSON line on stdout (rank 0).

`--impl reference` times the reference's own CPU path (the unmodified upstream package installed under baseline/_ref by
baseline/install_ref.sh; the oracle port only if that directory did not travel) on a bounded sample of the same workload.
The default run also carries short runs of the other BASELINE configs as `other_workloads`.

`--dump-outputs DIR` writes what the last timed step of the workload returned to its caller (rank 0): the loss as
DIR/loss.npy and every parameter's gradient as DIR/grad.<parameter name>.npy, float32, at most 64 MB in all (beyond that
the largest arrays are replaced by a fixed, seeded sample of their entries: see dump_outputs).  Weights and inputs are
seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "neural-process-family_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

WORKLOADS = {
    # name: (family, ctor kwargs, B per GPU, C, T, loss, description)
    "convcnp1d_b256_c128_t128": dict(family="ConvCNP", B=256, C=128, T=128, loss="cnpf",
                                     desc="BASELINE configs[1]: ConvCNP 1D default ctor, batch 256, 128 ctx / 128 tgt"),
    "cnp_b16_c32_t64": dict(family="CNP", B=16, C=32, T=64, loss="cnpf", desc="BASELINE configs[0]: CNP toy"),
    "attncnp_b64_c512_t512": dict(family="AttnCNP", B=64, C=512, T=512, loss="cnpf",
                                  desc="BASELINE configs[2]: AttnCNP transformer attention 512 ctx / 512 tgt"),
    "attncnp_b256_c512_t512": dict(family="AttnCNP", B=256, C=512, T=512, loss="cnpf",
                                   desc="BASELINE configs[2] at the SURVEY 8(d) batch: AttnCNP transformer attention 512 ctx / 512 tgt, 256 tasks"),
    "gridconvcnp_b128_32x32": dict(family="GridConvCNP", B=128, C=0, T=0, loss="cnpf",
                                   desc="BASELINE configs[3]: GridConvCNP 32x32x3, 128 images per GPU"),
    "gridconvlnp_b64_32x32_nz16": dict(family="GridConvLNP", B=64, C=0, T=0, loss="nll",
                                       desc="BASELINE configs[4]: GridConvLNP 32x32x3, 16 z samples, 64 images per GPU"),
}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d.get("bf16_tflops_sustained", d["bf16_tflops"]), source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1400.0, source="fallback")


# ----------------------------------------------------------------------------------------------------------------------
def make_model(family):
    import npf_b200
    from functools import partial
    from npf_b200.architectures import MLP, merge_flat_input
    torch.manual_seed(0)
    if family == "ConvCNP":
        return npf_b200.ConvCNP(1, 1)
    if family == "CNP":
        return npf_b200.CNP(1, 1)
    if family == "AttnCNP":
        return npf_b200.AttnCNP(1, 1, attention="transformer", XYEncoder=merge_flat_input(
            partial(MLP, n_hidden_layers=2, hidden_size=128), is_sum_merge=True))
    if family == "GridConvCNP":
        return npf_b200.GridConvCNP(1, 3)
    if family == "GridConvLNP":
        return npf_b200.GridConvLNP(1, 3, n_z_samples_train=16, is_q_zCct=False)
    raise ValueError(family)


def make_inputs(wl, B, seed, device="cpu", pin=False):
    g = torch.Generator().manual_seed(seed)
    if wl["family"].startswith("Grid"):
        img = torch.rand(B, 32, 32, 3, generator=g)
        mask = torch.zeros(B, 1024, dtype=torch.bool)
        for b in range(B):
            mask[b, torch.randperm(1024, generator=g)[:307]] = True
        t = dict(X_cntxt=mask.view(B, 32, 32, 1), Y_cntxt=img, X_trgt=torch.ones(B, 32, 32, 1, dtype=torch.bool),
                 Y_trgt=img.clone())
    else:
        C, T = wl["C"], wl["T"]
        t = dict(X_cntxt=torch.rand(B, C, 1, generator=g) * 2 - 1, Y_cntxt=torch.randn(B, C, 1, generator=g),
                 X_trgt=torch.rand(B, T, 1, generator=g) * 2 - 1, Y_trgt=torch.randn(B, T, 1, generator=g))
    if pin:
        t = {k: v.pin_memory() for k, v in t.items()}
    return {k: v.to(device) for k, v in t.items()} if device != "cpu" else t


class ClockSampler:
    """SM clock and clock-event (throttle) reasons sampled DURING the timed region: NVML in a background thread every
    ~2 ms (the graph-replayed timed region lasts tens of milliseconds, far shorter than one `nvidia-smi -lms` period);
    falls back to the nvidia-smi loop of the B200_PROFILING.md recipe if NVML cannot be loaded."""

    def __init__(self, index):
        self.index, self.samples, self.proc, self.nvml, self.stop_flag = index, [], None, None, False

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index())
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _physical_index(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [v.strip() for v in vis.split(",") if v.strip()]
            if self.index < len(ids) and ids[self.index].isdigit():
                return int(ids[self.index])
        return self.index

    def sample_now(self):
        """One synchronous sample from the caller's thread (the polling thread can be starved of the GIL by the launch loop)."""
        n = self.nvml
        if n is None:
            return
        try:
            mhz = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
            try:
                mask = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
            except Exception:
                mask = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
            bits = (n.nvmlClocksEventReasonHwSlowdown, n.nvmlClocksEventReasonHwThermalSlowdown, n.nvmlClocksEventReasonSwThermalSlowdown,
                    n.nvmlClocksEventReasonSwPowerCap)
            self.samples.append([str(mhz), str(self.max_mhz)] + ["Active" if mask & b else "Not Active" for b in bits])
        except Exception:
            pass

    def _poll(self):
        n = self.nvml
        names = (("hw_slowdown", n.nvmlClocksEventReasonHwSlowdown), ("hw_thermal_slowdown", n.nvmlClocksEventReasonHwThermalSlowdown),
                 ("sw_thermal_slowdown", n.nvmlClocksEventReasonSwThermalSlowdown), ("sw_power_cap", n.nvmlClocksEventReasonSwPowerCap))
        while not self.stop_flag:
            try:
                mhz = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
                try:
                    mask = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
                except Exception:
                    mask = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                self.samples.append([str(mhz), str(self.max_mhz)] + ["Active" if mask & bit else "Not Active" for _, bit in names])
            except Exception:
                pass
            time.sleep(0.002)

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append([s.strip() for s in line.split(",")])

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True
            self.thread.join(timeout=1.0)
        elif self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvml and nvidia-smi unavailable"], samples=0)
        else:
            self.proc.terminate()
        mhz = sorted(int(s[0]) for s in self.samples if s and s[0].isdigit())
        reasons = set()
        for s in self.samples:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        mx = [int(s[1]) for s in self.samples if len(s) > 1 and s[1].isdigit()]
        return dict(sm_mhz=mhz[len(mhz) // 2] if mhz else None, sm_max_mhz=max(mx) if mx else None, reasons=sorted(reasons),
                    samples=len(mhz), source="nvml" if self.nvml is not None else "nvidia-smi")


# ----------------------------------------------------------------------------------------------------------------------
REF_DIR = os.path.join(ROOT, "baseline", "_ref")          # the unmodified reference, installed by baseline/install_ref.sh
# tasks per CPU step (a bounded sample of the workload: the reference materialises [B,T,I,128] / [B,H,T,C] tensors)
CPU_SAMPLE_TASKS = {"ConvCNP": 8, "CNP": 16, "AttnCNP": 4, "GridConvCNP": 8, "GridConvLNP": 2}


def _reference_model(fam):
    """The reference's own model for the workload (npf.* from baseline/_ref), or None when it did not travel."""
    if not os.path.isdir(os.path.join(REF_DIR, "npf")):
        return None, None
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    try:
        import warnings
        warnings.filterwarnings("ignore")
        import npf
        from functools import partial
        from npf.architectures import MLP, merge_flat_input
    except Exception as e:                                                        # noqa: BLE001
        print(f"bench: reference import failed ({e}); falling back to the oracle port", file=sys.stderr)
        return None, None
    torch.manual_seed(0)
    if fam == "ConvCNP":
        m = npf.ConvCNP(1, 1)
    elif fam == "CNP":
        m = npf.CNP(1, 1)
    elif fam == "AttnCNP":
        m = npf.AttnCNP(1, 1, attention="transformer", XYEncoder=merge_flat_input(
            partial(MLP, n_hidden_layers=2, hidden_size=128), is_sum_merge=True))
    elif fam == "GridConvCNP":
        m = npf.GridConvCNP(1, 3)
    elif fam == "GridConvLNP":
        m = npf.GridConvLNP(1, 3, n_z_samples_train=16, is_q_zCct=False)
    else:
        raise ValueError(fam)
    return m.train(), npf


def cpu_reference_timing(wl, steps, warmup, budget_s=None):
    """The reference's CPU path on the host cores: fwd + loss + bwd of a bounded sample of the workload (Bc tasks per step,
    same C / T / image size as the GPU workload).  Times exactly `steps` steps, or with `budget_s` as many as fit in that many
    seconds (at least one, at most `steps`).  kind="reference": the unmodified upstream package (baseline/_ref, through
    its own public API: npf.<Model>(...)(X_cntxt, Y_cntxt, X_trgt, Y_trgt) -> npf.<Loss> -> backward); kind="port": the
    oracle's torch-CPU restatement, only when baseline/_ref did not travel."""
    avail = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    fam = wl["family"]
    Bc = min(CPU_SAMPLE_TASKS[fam], wl["B"])
    inp = make_inputs(wl, Bc, seed=1)
    Xc, Yc, Xt, Yt = inp["X_cntxt"], inp["Y_cntxt"], inp["X_trgt"], inp["Y_trgt"]
    ref_model, npf_ref = _reference_model(fam)
    if ref_model is not None:
        kind = "reference"
        crit = (npf_ref.CNPFLoss if wl["loss"] == "cnpf" else npf_ref.NLLLossLNPF)().train()

        def step():
            ref_model.zero_grad(set_to_none=True)
            crit(ref_model(Xc, Yc, Xt, Yt), Yt).backward()
        what = "unmodified reference package (baseline/_ref/npf), public API"
    else:
        kind = "port"
        from oracle import npf_oracle as O          # the one place bench.py may execute oracle/: the CPU arm
        model = make_model(fam)
        sd = {k: v.detach().clone().requires_grad_(v.is_floating_point()) for k, v in model.state_dict().items()}
        eps = torch.randn(16, Bc, 32, 32, 128) if fam == "GridConvLNP" else None

        def step():
            for v in sd.values():
                v.grad = None
            if fam == "ConvCNP":
                loc, scale = O.convcnp_forward(sd, Xc, Yc, Xt)
            elif fam == "CNP":
                loc, scale = O.cnp_forward(sd, Xc, Yc, Xt)
            elif fam == "AttnCNP":
                loc, scale = O.attncnp_forward(sd, Xc, Yc, Xt, attention="transformer")
            elif fam == "GridConvCNP":
                loc, scale = O.gridconvcnp_forward(sd, Xc, Yc)
            else:
                loc, scale, *_ = O.gridconvlnp_forward(sd, Xc, Yc, eps)
            (O.cnpf_loss(loc, scale, Yt) if wl["loss"] == "cnpf" else O.nll_lnpf_loss(loc, scale, Yt)).backward()
        what = "oracle/npf_oracle.py (torch-CPU restatement of the reference op sequence; baseline/_ref absent)"

    # all host threads are offered; ATen's broadcast-heavy kernels are not always fastest with all of them, so the thread
    # count is the best of {8 (the notebooks' N_THREADS), 16, 32, 64, all} on one step each -- the reference's best case
    t_cal = time.perf_counter()
    best = None
    for nt in sorted({n for n in (8, 16, 32, 64, avail) if n <= avail}):
        torch.set_num_threads(nt)
        step()
        t0 = time.perf_counter()
        step()
        dt = time.perf_counter() - t0
        if best is None or dt < best[0]:
            best = (dt, nt)
        if time.perf_counter() - t_cal > 40:
            break
    torch.set_num_threads(best[1])
    one = best[0]
    w = max(1, min(warmup, int(3.0 / max(one, 1e-3))))
    for _ in range(w - 1):
        step()
    k = steps if budget_s is None else max(1, min(steps, int(budget_s / max(one, 1e-3))))
    t0 = time.perf_counter()
    for _ in range(k):
        step()
    dt = (time.perf_counter() - t0) / k
    return dict(value=Bc / dt, unit="tasks/s", cores=torch.get_num_threads(), host_cpus=avail, kind=kind, tasks_per_step=Bc,
                sample=f"{k} steps of {Bc} tasks ({fam}, same C/T/image size as the GPU workload) in {dt * k:.1f}s; {what}; "
                       f"thread count = fastest of {{8,16,32,64,all}}"), dt * 1e3, k, w


# ----------------------------------------------------------------------------------------------------------------------
def make_loss(name, reduction="mean"):
    import npf_b200
    return dict(cnpf=npf_b200.CNPFLoss, nll=npf_b200.NLLLossLNPF, elbo=npf_b200.ELBOLossLNPF)[name](reduction=reduction)


def run_ours(wl_name, args, ctx, steps, warmup, full, capture_outputs=False):
    """One workload through the public API (GraphedStep): device-timed region with resident inputs, the end-to-end region
    from pinned host buffers, and the per-kernel breakdown.  `full` adds the fp32-path timing; `capture_outputs` returns the
    loss and the gradients of the last timed step as numpy arrays."""
    import npf_b200
    from npf_b200 import _cabi, ops
    from npf_b200.parallel import FlatGradients
    wl = WORKLOADS[wl_name]
    rank, world, dev, dist = ctx["rank"], ctx["world"], ctx["dev"], ctx["dist"]
    npf_b200.set_precision(args.precision)
    model = make_model(wl["family"]).to(dev).train()
    crit = make_loss(wl["loss"]).train()
    flat = FlatGradients(model, process_group=None if world == 1 else dist.group.WORLD)
    B = wl["B"]
    n_sets = 4
    dev_inputs = [make_inputs(wl, B, seed=100 * rank + i, device=dev) for i in range(n_sets)]
    host_inputs = [make_inputs(wl, B, seed=100 * rank + i, pin=True) for i in range(n_sets)]
    flush = ctx["flush"]

    def eager_step(inp):
        flat.zero_()
        out = model(inp["X_cntxt"], inp["Y_cntxt"], inp["X_trgt"], inp["Y_trgt"])
        loss = crit(out, inp["Y_trgt"])
        loss.backward()
        flat.all_reduce_mean()
        return loss

    # the public training-step API: the whole step recorded once into a CUDA graph and replayed (one host call per step)
    gstep = None if args.no_graph else npf_b200.GraphedStep(model, crit, flat=flat)

    def step(inp):
        if gstep is None:
            return eager_step(inp)
        return gstep(inp["X_cntxt"], inp["Y_cntxt"], inp["X_trgt"], inp["Y_trgt"])

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    warm = max(warmup, 3)
    for i in range(warm):
        step(dev_inputs[i % n_sets])
    barrier()

    # ---- timed region 1: inputs resident in HBM, CUDA events around every step, L2 flushed between steps ------------
    sampler = ClockSampler(ctx["local_rank"])
    if rank == 0:
        sampler.start()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    n0 = ops.launch_count()
    barrier()
    t_wall = time.perf_counter()
    timed = 0                               # steps the loop ran: what the rates below and the JSON line's `steps` count
    for i in range(steps):
        flush.fill_(float(i))
        evs[i][0].record()
        loss = step(dev_inputs[i % n_sets])
        evs[i][1].record()
        timed += 1
        if rank == 0 and i % 8 == 4:
            sampler.sample_now()            # under load: the GPU is several replays behind the host here
    barrier()
    t_wall = time.perf_counter() - t_wall
    launches = ops.launch_count() - n0 if gstep is None else gstep.last_launches * timed   # replays launch the recorded kernels
    dev_ms = sum(a.elapsed_time(b) for a, b in evs[:timed])
    clocks = sampler.stop() if rank == 0 else None
    outputs = None
    if capture_outputs:
        # what the caller of the last timed step received, copied before the regions below overwrite the loss and the gradients
        outputs = {"loss": loss.detach().float().cpu().numpy()}
        outputs.update({f"grad.{n}": p.grad.detach().float().cpu().numpy() for n, p in model.named_parameters() if p.grad is not None})

    # ---- timed region 2: end to end through the public API from pinned host buffers --------------------------------
    # Public API for host-resident batches: npf_b200.PipelinedStep(GraphedStep) -- every step copies its own inputs host -> device
    # (pinned buffers) and reads its own loss back; the copy of step i+1 and the read of step i-1 overlap step i's replay.
    pipe = None if gstep is None else npf_b200.PipelinedStep(gstep)

    def e2e_step(i):
        if pipe is None:
            inp = {k: v.to(dev, non_blocking=True) for k, v in host_inputs[i % n_sets].items()}
            return float(step(inp).item())
        return pipe.submit(host_inputs[i % n_sets])
    for i in range(3):
        e2e_step(i)
    if pipe is not None:
        pipe.drain()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for i in range(steps):
        e2e_step(i)              # host -> device copy of this step's inputs + device -> host read of a step's loss, every step
    if pipe is not None:
        pipe.drain()             # the last step's loss: K reads for K steps
    ev1.record()
    barrier()
    e2e_ms = ev0.elapsed_time(ev1)
    h2d = sum(v.numel() * v.element_size() for v in host_inputs[0].values())

    # ---- per-kernel CUDA-event breakdown (separate instrumented steps; events on the launching stream) --------------
    n_prof = min(steps, 10 if full else 4)
    _cabi.enable_timing(True)
    for i in range(n_prof):
        flush.fill_(0.0)
        eager_step(dev_inputs[i % n_sets])
    torch.cuda.synchronize()
    shaped = _cabi.collect_timing(by_shape=True)   # (name, bytes/call, flops/call) -> (total_ms, calls)
    _cabi.enable_timing(False)
    ktimes = {}
    for (name, nb, fl), (ms, n) in shaped.items():
        t = ktimes.get(name, (0.0, 0, 0, 0))
        ktimes[name] = (t[0] + ms, t[1] + n, t[2] + nb * n, t[3] + fl * n)

    # ---- the fp32 (FFMA) path of the same step, for reference next to the default precision -------------------------
    fp32_path = None
    if full and args.precision != "fp32":
        npf_b200.set_precision("fp32")
        g32 = None if args.no_graph else npf_b200.GraphedStep(model, crit, flat=flat)
        step32 = (lambda inp: eager_step(inp)) if g32 is None else (lambda inp: g32(inp["X_cntxt"], inp["Y_cntxt"], inp["X_trgt"], inp["Y_trgt"]))
        for i in range(3):
            step32(dev_inputs[i % n_sets])
        barrier()
        n32 = max(5, steps // 3)
        ev32 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n32)]
        for i in range(n32):
            flush.fill_(float(i))
            ev32[i][0].record()
            step32(dev_inputs[i % n_sets])
            ev32[i][1].record()
        barrier()
        ms32 = sum(a.elapsed_time(b) for a, b in ev32) / n32
        fp32_path = dict(ms_per_step=ms32, value=B * world / (ms32 * 1e-3), unit="tasks/s", steps=n32, note="same step with precision=fp32 (FFMA GEMMs), rank-local time")
        npf_b200.set_precision(args.precision)
        del g32

    tot = torch.tensor([dev_ms, e2e_ms], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(tot, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms = float(tot[0]), float(tot[1])
    flat.detach()
    del gstep, model, flat, dev_inputs, host_inputs
    torch.cuda.empty_cache()
    tasks = B * world * timed
    return dict(wl=wl, B=B, steps=timed, warmup=warm, value=tasks / (dev_ms * 1e-3), ms_per_step=dev_ms / timed,
                e2e=dict(value=B * world * steps / (e2e_ms * 1e-3), unit="tasks/s", h2d_bytes_per_step=h2d, d2h_bytes_per_step=4),
                launches=launches, wall_ms_per_step=t_wall * 1e3 / timed, clocks=clocks, ktimes=ktimes, shaped=shaped, n_prof=n_prof,
                fp32_path=fp32_path, outputs=outputs)


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, outputs, limit_bytes=DUMP_LIMIT_BYTES):
    """Writes every array as out_dir/<name>.npy in float32, at most `limit_bytes` in all.  When the arrays hold more, the
    largest ones are cut to a common number of entries: a sample drawn at seeded positions (the same on every run) from the
    flattened array, kept in index order, so two runs still compare entry for entry; smaller arrays stay whole."""
    import numpy as np
    arrays = {name: np.asarray(a, dtype=np.float32) for name, a in outputs.items()}
    budget = (limit_bytes - 128 * len(arrays)) // 4          # float32 entries, after one 128-byte .npy header per file
    cap = None
    if sum(a.size for a in arrays.values()) > budget:
        sizes = sorted(a.size for a in arrays.values())
        for i, n in enumerate(sizes):
            share = budget // (len(sizes) - i)
            if n > share:
                cap = share
                break
            budget -= n
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if cap is not None and a.size > cap:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, cap, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def workload_config(name, world, no_graph):
    wl = WORKLOADS[name]
    return dict(workload=name, description=wl["desc"], tasks_per_gpu=wl["B"], global_batch=wl["B"] * max(world, 1),
                n_cntxt=wl["C"], n_trgt=wl["T"], parallelism=f"dp{max(world, 1)} (tasks sharded, flat-gradient all-reduce)",
                l2="flushed between timed steps (256 MiB write, outside the per-step event pairs)",
                launch="eager" if no_graph else "cuda graph replay (npf_b200.GraphedStep)")


# ----------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100, help="number of timed steps")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="convcnp1d_b256_c128_t128", choices=list(WORKLOADS))
    ap.add_argument("--precision", default="bf16x3", choices=["fp32", "bf16", "bf16x3"],
                    help="bf16x3 (default): tcgen05 linear layers with 3-term split-bf16 operands, fp32 accumulate -- meets the fp32 parity bar (1e-4); "
                         "fp32: FFMA GEMMs; bf16: single-pass bf16 operands (1e-2 bar)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-others", action="store_true", help="skip the short runs of the other BASELINE workloads (`other_workloads`)")
    ap.add_argument("--no-graph", action="store_true", help="eager launches instead of the CUDA-graph replay of the step (npf_b200.GraphedStep)")
    ap.add_argument("--kernel-times", action="store_true", help="print the per-kernel CUDA-event breakdown to stderr")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the loss and the gradients of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    wl = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        if rank != 0:
            return
        cb, ms, k, w = cpu_reference_timing(wl, args.steps, args.warmup)
        cfg = dict(workload=args.workload, description=wl["desc"], tasks_per_gpu=wl["B"], global_batch=wl["B"] * max(args.gpus, 1),
                   n_cntxt=wl["C"], n_trgt=wl["T"], cpu_sample_tasks_per_step=cb["tasks_per_step"],
                   note=f"CPU arm: each step is a bounded sample of {cb['tasks_per_step']} tasks of the workload (the GPU arm runs {wl['B']} per GPU); "
                        "tasks/s is per-task cost and extrapolates linearly in the batch")
        line = dict(impl="reference", metric="tasks/sec (meta-batch fwd+bwd)", value=cb["value"], unit="tasks/s",
                    n_gpus=args.gpus, steps=k, warmup=w, ms_per_step=ms, higher_is_better=True, scaling="weak",
                    vs_baseline=None, dtype="f32", data="synthetic", config=cfg, cpu_baseline=cb,
                    e2e=dict(value=cb["value"], unit="tasks/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
        print(json.dumps(line))
        return

    import npf_b200  # noqa: F401

    assert torch.cuda.is_available(), "bench.py (impl=ours) needs a GPU; there is no CPU fallback"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    ctx = dict(rank=rank, world=world, local_rank=local_rank, dev=dev, dist=dist,
               flush=torch.empty(256 * 1024 * 1024 // 4, device=dev))
    peaks = measured_peaks()

    r = run_ours(args.workload, args, ctx, args.steps, args.warmup, full=True, capture_outputs=bool(args.dump_outputs))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, r["outputs"])
    # short runs of the other BASELINE workloads, so that one driver-run line shows every config (same protocol, fewer steps)
    others = {}
    if not args.no_others and args.workload == "convcnp1d_b256_c128_t128":
        for name in ("cnp_b16_c32_t64", "attncnp_b64_c512_t512", "gridconvcnp_b128_32x32", "gridconvlnp_b64_32x32_nz16"):
            o = run_ours(name, args, ctx, steps=max(5, min(args.steps, 20) // 2), warmup=3, full=False)
            if rank == 0:
                roof_o, _ = roofline(o["wl"], o["ktimes"], o["n_prof"], o["B"], peaks, o["shaped"])
                others[name] = dict(value=o["value"], unit="tasks/s", ms_per_step=o["ms_per_step"], steps=o["steps"], warmup=o["warmup"],
                                    e2e=o["e2e"], gpu_launches=o["launches"], config=workload_config(name, world, args.no_graph),
                                    roofline=roof_o,
                                    kernel_ms_per_step={k: round(v[0] / o["n_prof"], 4) for k, v in sorted(o["ktimes"].items(), key=lambda kv: -kv[1][0])[:8]})
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    ktimes, n_prof = r["ktimes"], r["n_prof"]
    roof, roof_table = roofline(wl, ktimes, n_prof, r["B"], peaks, r["shaped"])
    line = dict(metric="tasks/sec (meta-batch fwd+bwd)", value=r["value"], unit="tasks/s", n_gpus=world, steps=r["steps"],
                warmup=r["warmup"], ms_per_step=r["ms_per_step"], higher_is_better=True, scaling="weak",
                vs_baseline=None, dtype={"fp32": "f32", "bf16": "bf16", "bf16x3": "bf16x3 (fp32-equivalent)"}[args.precision],
                data="synthetic", config=workload_config(args.workload, world, args.no_graph), clocks=r["clocks"],
                e2e=r["e2e"], gpu_launches=r["launches"], wall_ms_per_step=r["wall_ms_per_step"], roofline=roof, kernel_rooflines=roof_table,
                kernel_ms_per_step={k: round(v[0] / n_prof, 4) for k, v in sorted(ktimes.items(), key=lambda kv: -kv[1][0])},
                kernel_timing="per-call CUDA events on the launching stream in 10 instrumented eager steps after the timed region "
                              "(the timed region itself replays a CUDA graph: no per-kernel events inside it)")
    if r["fp32_path"] is not None:
        line["fp32_path"] = r["fp32_path"]
    if others:
        line["other_workloads"] = others
    if not args.no_cpu_baseline:
        cb, _, _, _ = cpu_reference_timing(wl, 200, 2, budget_s=15.0)
        line["cpu_baseline"] = cb
    if args.kernel_times:
        for k, v in sorted(ktimes.items(), key=lambda kv: -kv[1][0]):
            print(f"  {k:28s} {v[0] / n_prof:9.4f} ms/step  {v[1] // n_prof:4d} calls/step", file=sys.stderr)
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


def roofline(wl, ktimes, n_prof, B, peaks, shaped):
    """Roofline of the dominant kernel = the (C-ABI entry point, problem size) class with the largest share of the step,
    plus aggregate figures for every timed entry point.  achieved = algorithmic bytes of ONE launch (SURVEY.md section 8d:
    every operand and result once, fp32; table in npf_b200/_cabi.py) / the average duration of that launch, measured with
    CUDA events on the launching stream; peak = MEASURED_PEAKS.json (sustained figures: the kernels run inside a long
    step); traffic = DRAM bytes of the same launch from the committed `ncu --set full` capture (profiles/traffic_r2.json)."""
    if not ktimes:
        return None, None
    total = sum(v[0] for v in ktimes.values())
    table = {}

    def entry(ms, calls, nbytes, flops):
        gbs = nbytes / (ms * 1e-3) / 1e9
        tfs = flops / (ms * 1e-3) / 1e12
        # the binding roof: whichever of HBM / tensor time is longer for this op mix
        t_hbm, t_tc = nbytes / (peaks["hbm_gbs"] * 1e9), flops / (peaks["bf16_tflops"] * 1e12)
        bound = "hbm" if t_hbm >= t_tc else "tensor"
        return dict(bound=bound, achieved=gbs if bound == "hbm" else tfs, peak=peaks["hbm_gbs"] if bound == "hbm" else peaks["bf16_tflops"],
                    unit="GB/s" if bound == "hbm" else "TFLOP/s", frac=(gbs / peaks["hbm_gbs"]) if bound == "hbm" else tfs / peaks["bf16_tflops"],
                    launches_per_step=calls // n_prof, ms_per_step=ms / n_prof, share_of_step=ms / total, gbytes_per_s=gbs, tflops=tfs)

    for name, (ms, calls, nbytes, flops) in ktimes.items():
        if nbytes:
            table[name] = entry(ms, calls, nbytes, flops)
    classes = {k: v for k, v in shaped.items() if k[1]}
    if not classes:
        return None, table or None
    (name, nb, fl), (ms, calls) = max(classes.items(), key=lambda kv: kv[1][0])
    e = entry(ms, calls, nb * calls, fl * calls)
    traffic, cuda_kernel = None, None
    for fn in ("traffic_r2.json", "traffic_r1.json"):      # dram__bytes_read.sum + dram__bytes_write.sum of one launch (ncu --set full captures)
        try:
            with open(os.path.join(ROOT, "profiles", fn)) as f:
                for rec in json.load(f)["kernels"]:
                    if rec["entry"] == name and rec.get("algorithmic_bytes") in (None, nb) and traffic is None:
                        traffic, cuda_kernel = rec["dram_bytes"], rec["cuda_kernel"]
        except (OSError, KeyError, ValueError):
            pass
    dom = dict(kernel=name, cuda_kernel=cuda_kernel, algorithmic_bytes_per_launch=nb, flops_per_launch=fl, peak_source=peaks["source"], traffic=traffic,
               avg_launch_ms=ms / calls, **{k: e[k] for k in ("bound", "achieved", "peak", "unit", "frac", "launches_per_step", "share_of_step")})
    return dom, table


if __name__ == "__main__":
    main()
