"""Data parallelism over tasks: every rank owns a contiguous shard of the meta-batch and a replica of the parameters;
the only exchange is ONE all-reduce of a flat fp32 gradient buffer per step (SURVEY.md section 8e).

``FlatGradients`` allocates one contiguous buffer and makes every ``p.grad`` a view into it, so the backward kernels'
results land in the bucket directly and the collective is a single NCCL call (0.5-2 MB: latency-bound on NVLink 5 /
NVSwitch).  Works with any ``torch.distributed`` backend (``gloo`` on CPU for the host-logic tests)."""
import torch
import torch.distributed as dist

__all__ = ["FlatGradients", "FlatAdam", "P2PAllReduce", "shard_tasks", "sync_batchnorm_", "sync_moments"]


class _DevMem:
    """A cudaMalloc allocation of the library (npf_p2p_alloc) exposed to torch through __cuda_array_interface__ (zero copy)."""

    def __init__(self, ptr, numel, typestr):
        self.ptr, self.numel = ptr, numel
        self.__cuda_array_interface__ = dict(shape=(numel,), typestr=typestr, data=(ptr, False), version=2)


class P2PAllReduce:
    """One-kernel mean all-reduce of the flat gradient bucket over NVLink peer memory (csrc/p2p.cu): every rank maps the other
    ranks' buckets (CUDA IPC, one process per GPU of one node) and reads them directly; inter-rank barriers are epoch flags in peer
    memory inside the kernel.  ``bucket`` is the tensor the gradients are accumulated into (allocated here so that it can be shared);
    ``reduce_()`` leaves the mean in it."""

    def __init__(self, numel, device, group=None):
        import ctypes
        from . import _cabi
        self.group, self.rank, self.world = group, dist.get_rank(group), dist.get_world_size(group)
        n = (numel + 3) // 4 * 4
        self.n = n
        mine = []
        for nbytes in (4 * n, 4 * n, 4 * 2 * self.world, 8):          # bucket, output, signal block, local state
            p = ctypes.c_void_p()
            _cabi.call("npf_p2p_alloc", ctypes.byref(p), nbytes)
            mine.append(p.value)
        self._mine = mine
        torch.cuda.synchronize(device)
        handles = []
        for ptr in (mine[0], mine[2], mine[1]):
            h = (ctypes.c_ubyte * 64)()
            _cabi.call("npf_p2p_get_handle", ptr, h)
            handles.append(bytes(h))
        gathered = [None] * self.world
        dist.all_gather_object(gathered, (handles, torch.cuda.current_device()), group=group)
        self._opened, ins, sigs, outs = [], [], [], []
        for r, (hs, _dev) in enumerate(gathered):
            if r == self.rank:
                ins.append(mine[0]); sigs.append(mine[2]); outs.append(mine[1])
                continue
            ptrs = []
            for hb in hs:
                p = ctypes.c_void_p()
                _cabi.call("npf_p2p_open", (ctypes.c_ubyte * 64).from_buffer_copy(hb), ctypes.byref(p))
                ptrs.append(p.value)
                self._opened.append(p.value)
            ins.append(ptrs[0]); sigs.append(ptrs[1]); outs.append(ptrs[2])
        self._in = (ctypes.c_void_p * self.world)(*ins)
        self._sig = (ctypes.c_void_p * self.world)(*sigs)
        self._out = (ctypes.c_void_p * self.world)(*outs)
        # two-shot (each rank reduces one slice and writes it to everybody) from 4 ranks up, one-shot (everybody reads everything) below:
        # measured on B200 NVLink, profiles/r2/allreduce_placement.md
        self.two_shot = self.world >= 4
        self.bucket = torch.as_tensor(_DevMem(mine[0], n, "<f4"), device=device)
        self.out = torch.as_tensor(_DevMem(mine[1], n, "<f4"), device=device)
        dist.barrier(group=group)                                          # every rank has opened every handle before the first launch

    def close(self):
        """Unmap the peers' allocations and free this rank's (collective: every rank calls it; nobody may still be inside an all-reduce)."""
        from . import _cabi
        if self._mine is None:
            return
        torch.cuda.synchronize()
        dist.barrier(group=self.group)
        for ptr in self._opened:
            _cabi.call("npf_p2p_close", ptr)
        dist.barrier(group=self.group)                  # every peer has unmapped before the owner frees
        self.bucket = self.out = None
        for ptr in self._mine:
            _cabi.call("npf_p2p_free", ptr)
        self._mine, self._opened = None, []

    def reduce_(self):
        from . import _cabi
        if self.two_shot:
            _cabi.call("npf_allreduce_mean_p2p2", self._in, self._sig, self._out, self._mine[3], self.rank, self.world, self.n,
                       torch.cuda.current_stream().cuda_stream)
        else:
            _cabi.call("npf_allreduce_mean_p2p", self._in, self._sig, self._mine[1], self._mine[3], self.rank, self.world, self.n,
                       torch.cuda.current_stream().cuda_stream)
        self.bucket.copy_(self.out)
        return self.bucket


def _try_p2p(numel, device, group):
    """P2PAllReduce if every rank of the group can set it up (same node, peer access), else None -- decided collectively."""
    if device.type != "cuda" or dist.get_backend(group) != "nccl":
        return None
    p2p, ok = None, 1
    try:
        p2p = P2PAllReduce(numel, device, group)
    except Exception:                                                       # noqa: BLE001  (IPC / peer access unavailable)
        ok = 0
    flag = torch.tensor([ok], device=device, dtype=torch.int32)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
    return p2p if int(flag.item()) == 1 else None


class FlatGradients:
    def __init__(self, module, process_group=None):
        self.params = [p for p in module.parameters() if p.requires_grad]
        self.group = process_group
        # every parameter's slice starts on a 128-byte boundary (vectorised / float4-atomic gradient kernels need 16 B)
        self.offsets, n = [], 0
        for p in self.params:
            self.offsets.append(n)
            n += (p.numel() + 31) // 32 * 32
        dev = self.params[0].device if self.params else torch.device("cpu")
        self.p2p = None
        if dev.type == "cuda" and dist.is_available() and dist.is_initialized() and dist.get_world_size(process_group) > 1:
            self.p2p = _try_p2p(n, dev, process_group)          # one-kernel all-reduce over NVLink peer memory (falls back to NCCL)
        self.flat = self.p2p.bucket[:n] if self.p2p is not None else torch.zeros(n, dtype=torch.float32, device=dev)
        self._attach()

    def _attach(self):
        base = self.flat.data_ptr()
        for p, off in zip(self.params, self.offsets):
            p.grad = self.flat[off: off + p.numel()].view_as(p)
            # the weight-gradient kernels add straight into the bucket for THESE parameters only (ops._gbuf)
            p._npf_direct_grad = p.is_cuda
        self._grad_ptrs = [base + 4 * off for off in self.offsets]

    def detach(self):
        """Give the parameters back to plain autograd accumulation (drops the views into the bucket) and release the peer-memory
        all-reduce, if any (collective on more than one rank)."""
        for p in self.params:
            p._npf_direct_grad = False
            p.grad = None
        if self.p2p is not None:
            self.flat = None
            self.p2p.close()
            self.p2p = None

    def zero_(self):
        """Zero the bucket (one memset) and re-attach the views if anything dropped or replaced one of them
        (``optimizer.zero_grad(set_to_none=True)``, ``model.zero_grad()``, a ``.to()`` of the module)."""
        self.flat.zero_()
        for p, ptr in zip(self.params, self._grad_ptrs):
            g = p.grad
            if g is None or g.data_ptr() != ptr:
                self._attach()
                break

    @property
    def world_size(self):
        if self.group is None and not (dist.is_available() and dist.is_initialized()):
            return 1
        return dist.get_world_size(self.group)

    def all_reduce_mean(self):
        """grad <- mean over ranks of the per-rank (local-batch-mean) gradients: equals the gradient of the global
        batch mean for equal shards.  No-op on a single rank."""
        w = self.world_size
        if w == 1:
            return self.flat
        if self.p2p is not None:
            self.p2p.reduce_()
            return self.flat
        if self.flat.is_cuda:      # NCCL averages inside the collective: no separate 1/G kernel
            dist.all_reduce(self.flat, op=dist.ReduceOp.AVG, group=self.group)
        else:                      # gloo (CPU host-logic tests) has no AVG
            dist.all_reduce(self.flat, op=dist.ReduceOp.SUM, group=self.group)
            self.flat.mul_(1.0 / w)
        return self.flat


class FlatAdam:
    """torch.optim.Adam (the optimizer of upstream utils/train.py:50) over the flat gradient bucket: the parameters are
    re-pointed into ONE contiguous fp32 buffer laid out like ``flat`` (same 128-byte aligned slots), so a step is a single
    elementwise kernel (``npf_adam_step``) over (param, grad, exp_avg, exp_avg_sq) instead of ~40 small foreach launches.
    ``lr`` may be changed between steps (``opt.lr = ...``: ExponentialLR is ``opt.lr *= gamma`` per epoch);
    ``grad_scale`` pre-multiplies the gradient (1 / world size); ``max_grad_norm`` clips by the global norm like
    ``torch.nn.utils.clip_grad_norm_`` (skorch ``GradientNormClipping`` of the latent notebooks) with the norm reduced and
    consumed on the device (``npf_sqnorm`` + ``npf_adam_step_clipped``): no host sync, capturable in a CUDA graph."""

    def __init__(self, flat, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0):
        self.flat, self.lr, self.betas, self.eps, self.weight_decay = flat, lr, betas, eps, weight_decay
        self.step_count = 0
        g = flat.flat
        self.param = torch.zeros_like(g)
        with torch.no_grad():
            for p, off in zip(flat.params, flat.offsets):
                view = self.param[off: off + p.numel()].view_as(p)
                view.copy_(p.data)
                p.data = view                     # the module now reads / the kernels now update the flat storage
        self.exp_avg = torch.zeros_like(g)
        self.exp_avg_sq = torch.zeros_like(g)
        self._sqnorm = torch.zeros(1, dtype=torch.float32, device=g.device)

    def last_grad_norm(self):
        """Global gradient norm seen by the last clipped step (device scalar; reading it synchronises)."""
        return self._sqnorm.sqrt()

    def global_grad_norm(self):
        return self.flat.flat.norm()              # padding between slots is zero

    def step(self, grad_scale=1.0, max_grad_norm=None):
        from . import _cabi
        if not self.param.is_cuda:
            raise RuntimeError("FlatAdam: CUDA only (there is no CPU fallback)")
        self.step_count += 1
        n = self.param.numel()
        if max_grad_norm is not None:
            st = torch.cuda.current_stream().cuda_stream
            _cabi.call("npf_sqnorm", self.flat.flat.data_ptr(), n, self._sqnorm.data_ptr(), st)
            _cabi.call("npf_adam_step_clipped", self.param.data_ptr(), self.flat.flat.data_ptr(), self.exp_avg.data_ptr(),
                       self.exp_avg_sq.data_ptr(), n, self.step_count, float(self.lr), float(self.betas[0]), float(self.betas[1]),
                       float(self.eps), float(self.weight_decay), float(grad_scale), self._sqnorm.data_ptr(), float(max_grad_norm), st)
            return
        if self.param.is_cuda:
            _cabi.call("npf_adam_step", self.param.data_ptr(), self.flat.flat.data_ptr(), self.exp_avg.data_ptr(), self.exp_avg_sq.data_ptr(), n,
                       self.step_count, float(self.lr), float(self.betas[0]), float(self.betas[1]), float(self.eps), float(self.weight_decay),
                       float(grad_scale), torch.cuda.current_stream().cuda_stream)
            return
        raise RuntimeError("FlatAdam: CUDA only (there is no CPU fallback)")

    def state_dict(self):
        return dict(step=self.step_count, lr=self.lr, exp_avg=self.exp_avg.clone(), exp_avg_sq=self.exp_avg_sq.clone())

    # ---- interchange with torch.optim.Adam (the ``optimizer.pt`` upstream's skorch Checkpoint writes next to ``params.pt``)
    def torch_state_dict(self):
        """The state in ``torch.optim.Adam.state_dict()`` layout (per-parameter moments, index keys, one param group)."""
        state = {}
        for i, (p, off) in enumerate(zip(self.flat.params, self.flat.offsets)):
            sl = slice(off, off + p.numel())
            state[i] = dict(step=torch.tensor(float(self.step_count)), exp_avg=self.exp_avg[sl].view_as(p).detach().cpu().clone(),
                            exp_avg_sq=self.exp_avg_sq[sl].view_as(p).detach().cpu().clone())
        group = dict(lr=self.lr, betas=tuple(self.betas), eps=self.eps, weight_decay=self.weight_decay, amsgrad=False,
                     params=list(range(len(self.flat.params))))
        return dict(state=state, param_groups=[group])

    def load_torch_state_dict(self, sd):
        """Resume from a ``torch.optim.Adam`` state dict -- current index-keyed layout or the legacy id-keyed one of the
        upstream checkpoints: the i-th entry of ``param_groups[0]['params']`` belongs to the i-th parameter."""
        groups = sd["param_groups"]
        if len(groups) != 1:
            raise ValueError("FlatAdam.load_torch_state_dict: exactly one param group expected")
        g, keys = groups[0], groups[0]["params"]
        if len(keys) != len(self.flat.params):
            raise ValueError(f"optimizer state has {len(keys)} parameters, the model {len(self.flat.params)}")
        if g.get("amsgrad", False):
            raise NotImplementedError("FlatAdam: amsgrad state is not supported")
        steps = set()
        for key, p, off in zip(keys, self.flat.params, self.flat.offsets):
            st = sd["state"].get(key)
            if st is None:        # parameter never stepped
                continue
            if tuple(st["exp_avg"].shape) != tuple(p.shape):
                raise ValueError(f"optimizer state shape {tuple(st['exp_avg'].shape)} does not match parameter {tuple(p.shape)}")
            sl = slice(off, off + p.numel())
            self.exp_avg[sl].copy_(st["exp_avg"].reshape(-1))
            self.exp_avg_sq[sl].copy_(st["exp_avg_sq"].reshape(-1))
            steps.add(int(st["step"]))
        if len(steps) > 1:
            raise ValueError(f"FlatAdam keeps one step count for all parameters, the state has {sorted(steps)}")
        self.step_count = steps.pop() if steps else 0
        self.lr, self.betas = float(g["lr"]), tuple(g["betas"])
        self.eps, self.weight_decay = float(g["eps"]), float(g["weight_decay"])

    def load_state_dict(self, sd):
        self.step_count, self.lr = int(sd["step"]), float(sd["lr"])
        self.exp_avg.copy_(sd["exp_avg"])
        self.exp_avg_sq.copy_(sd["exp_avg_sq"])


class _AllReduceSum(torch.autograd.Function):
    """Differentiable sum-all-reduce: the gradient of a sum over ranks is the sum over ranks of the gradients."""

    @staticmethod
    def forward(ctx, t, group):
        ctx.group = group
        out = t.detach().clone()
        dist.all_reduce(out, op=dist.ReduceOp.SUM, group=group)
        return out

    @staticmethod
    def backward(ctx, g):
        g = g.contiguous().clone()
        dist.all_reduce(g, op=dist.ReduceOp.SUM, group=ctx.group)
        return g, None


def sync_moments(mean, var, n_local, group=None):
    """Per-rank batch statistics (mean, biased var over ``n_local`` positions) -> statistics of the GLOBAL batch, by ONE
    all-reduce of the 2C + 1 numbers (sum x, sum x^2, count) per BatchNorm layer in forward and one of their gradients in
    backward (SURVEY.md section 8e caveat).  Returns (mean, var, n_total); differentiable."""
    C = mean.numel()
    packed = torch.cat([mean * n_local, (var + mean * mean) * n_local, mean.new_full((1,), float(n_local))])
    tot = _AllReduceSum.apply(packed, group)
    n = tot[2 * C]
    g_mean = tot[:C] / n
    g_var = tot[C:2 * C] / n - g_mean * g_mean
    return g_mean, g_var, n


def sync_batchnorm_(module, group=None):
    """Mark every BatchNorm of ``module`` (the ``Normalization=nn.BatchNorm*`` CNNs of the notebooks) as synchronised over
    ``group``: in train mode the folded pre-activation affine then uses the statistics of the global meta-batch, which
    makes an N-rank run equal to the single-process reference on the same global batch (without it every rank normalises
    with its own shard: "replicas with local BN").  In place; returns the module.  Eval mode is unaffected."""
    for m in module.modules():
        if isinstance(m, (torch.nn.BatchNorm1d, torch.nn.BatchNorm2d)):
            m._npf_sync_group = (group,)
    return module


def shard_tasks(batch, rank, world_size):
    """Contiguous split of the task axis: rank g gets tasks [g*B/G, (g+1)*B/G).  ``batch`` is a dict of tensors whose
    first axis is the task axis; B must be divisible by the world size."""
    out = {}
    for k, v in batch.items():
        B = v.shape[0]
        if B % world_size:
            raise ValueError(f"meta-batch {B} is not divisible by world size {world_size}")
        s = B // world_size
        out[k] = v[rank * s: (rank + 1) * s]
    return out
