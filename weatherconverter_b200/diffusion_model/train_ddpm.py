"""Denoising-loss training with the reference's step semantics (diffusion_model/train_ddpm.py:71-133) on libwc_b200.so.

The reference step is
    noise = randn_like(images); t = randint(0, T, (B,)); noisy = scheduler.add_noise(images, noise, t)
    loss = MSELoss(model(noisy, t), noise); loss.backward(); Adam.step()                      (:95-114)
Here the forward, the loss, the whole backward and the Adam update run as static launch plans of hand-written kernels
(csrc/unet_train.cu); PyTorch only owns the memory, the streams and, for more than one GPU, the NCCL communicator.

Data parallelism (SURVEY 8e; the reference itself is single-GPU): one process per GPU, each with a full replica and
its own mini-batch; gradients are summed with NCCL all-reduces issued per bucket as soon as the backward plan has
finished the bucket's parameters (the flat gradient buffer is laid out in backward-completion order so that every
bucket is one contiguous slice), then every rank applies the same fused Adam update with the 1/world scale folded in.

``train()`` takes that fused path for the reference's own pair (``nn.MSELoss()`` + plain ``torch.optim.Adam``) and runs
the reference's step body on the differentiable ``Unet`` (models/unet_base.py) for any other criterion and optimizer.
"""
import ctypes as C

import torch
import torch.distributed as dist

from .. import _lib
from .._lib import check, lib, ptr, stream_ptr
from .._plans import PlanHandle, c_tensor_args
from .models.unet_base import Unet

device = torch.device("cuda" if torch.cuda.is_available() else "cpu")


def _backward_group(name: str, n_ups: int, n_mids: int, n_downs: int) -> int:
    """Coarse backward-completion rank of a parameter (conv_out first ... conv_in, then the time-embedding path, whose
    gradients are only complete after every ResNet block has contributed)."""
    if "t_emb_layers" in name or name.startswith("t_proj"):
        return 3 + n_ups + n_mids + n_downs
    head = name.split(".")
    if head[0] in ("conv_out", "norm_out"):
        return 0
    if head[0] == "ups":
        return 1 + (n_ups - 1 - int(head[1]))
    if head[0] == "mids":
        return 1 + n_ups + (n_mids - 1 - int(head[1]))
    if head[0] == "downs":
        return 1 + n_ups + n_mids + (n_downs - 1 - int(head[1]))
    if head[0] == "conv_in":
        return 1 + n_ups + n_mids + n_downs
    raise KeyError(name)


def make_buckets(names, slices, groups, ready, n_ops, used, bucket_bytes):
    """Contiguous [start, stop) slices of the flat gradient buffer + the backward-op count after which each is final.
    A bucket is closed at a block boundary (change of backward group) once it holds >= bucket_bytes."""
    buckets, start, cur_group, cur_ready = [], 0, groups[0], 0
    for i, name in enumerate(names):
        off, _ = slices[name]
        if groups[i] != cur_group and (off - start) * 4 >= bucket_bytes:
            buckets.append((start, off, cur_ready))
            start, cur_ready = off, 0
        cur_group = groups[i]
        cur_ready = max(cur_ready, ready[i])
    buckets.append((start, used, max(cur_ready, n_ops)))
    fixed, hi = [], 0
    for (a, b, r) in buckets:      # op counts must not decrease from bucket to bucket
        hi = max(hi, r)
        fixed.append((a, b, hi))
    return fixed


def backward_with_buckets(run_ops, n_ops, flat_grads, buckets, world, group=None):
    """Run the backward plan slice by slice; as soon as a bucket's gradients are final, start its all-reduce (async: NCCL
    runs it on its own stream, ordered after the work already queued on the current stream) and keep computing."""
    works, cursor = [], 0
    for (a, b, upto) in buckets:
        if upto > cursor:
            run_ops(cursor, upto)
            cursor = upto
        if world > 1:
            works.append(dist.all_reduce(flat_grads[a:b], op=dist.ReduceOp.SUM, group=group, async_op=True))
    if cursor < n_ops:
        run_ops(cursor, n_ops)
    for w in works:
        w.wait()


class DenoisingTrainer:
    """Owns flat fp32 parameter / gradient / Adam-moment buffers (the model's parameters become views into the flat
    parameter buffer) and the C training plan bound to one (batch, H, W), held as a ``_plans.PlanHandle``."""

    def __init__(self, model: Unet, scheduler, lr=1e-4, betas=(0.9, 0.999), eps=1e-8, process_group=None,
                 bucket_bytes=64 << 20, seed=None, data_parallel=True):
        if not torch.cuda.is_available():
            raise RuntimeError("wc_b200 training needs a CUDA device (sm_100a); there is no CPU fallback")
        self.model, self.scheduler = model, scheduler
        self.lr, self.betas, self.eps = float(lr), (float(betas[0]), float(betas[1])), float(eps)
        self.group = process_group
        # data_parallel=False: a single-process trainer inside an initialised process group (no broadcast, no all-reduce) - e.g.
        # the one-process reference run of tools/ddp_check.py; constructing a data-parallel trainer is a COLLECTIVE call
        self.world = (dist.get_world_size(process_group)
                      if (data_parallel and dist.is_available() and dist.is_initialized()) else 1)
        self.rank = dist.get_rank(process_group) if self.world > 1 else 0
        self.bucket_bytes = int(bucket_bytes)
        self.step_count = 0
        named = list(model.named_parameters())
        dev = named[0][1].device
        if dev.type != "cuda":
            raise RuntimeError("move the model to the GPU before building a DenoisingTrainer")
        n_levels = len(model.down_channels) - 1
        n_mids = len(model.mid_channels) - 1
        order = sorted(range(len(named)), key=lambda i: (_backward_group(named[i][0], n_levels, n_mids, n_levels), i))
        total = sum((p.numel() + 3) & ~3 for _, p in named)   # every tensor starts 16-byte aligned
        self.flat_params = torch.zeros(total, device=dev, dtype=torch.float32)   # zeros: the alignment gaps are stepped by Adam too
        self.flat_grads = torch.zeros(total, device=dev, dtype=torch.float32)
        self.exp_avg = torch.zeros(total, device=dev, dtype=torch.float32)
        self.exp_avg_sq = torch.zeros(total, device=dev, dtype=torch.float32)
        self.slices, self.groups = {}, []
        off = 0
        for i in order:
            name, p = named[i]
            n = p.numel()
            off = (off + 3) & ~3          # 16-byte alignment of every tensor
            view = self.flat_params[off:off + n].view(p.shape)
            view.copy_(p.data)
            p.data = view
            p.grad = self.flat_grads[off:off + n].view(p.shape)
            self.slices[name] = (off, n)
            self.groups.append(_backward_group(name, n_levels, n_mids, n_levels))
            off += n
        self.used = off
        self.names = [named[i][0] for i in order]
        self._plan = None            # PlanHandle of the training plan, made by the first _bind
        self._bound = None
        self._buckets = []
        self._keep = None
        self.loss = torch.zeros(1, device=dev, dtype=torch.float32)
        # Replicas must start identical (what torch DDP guarantees by broadcasting rank 0's parameters at construction):
        # do not rely on every rank having seeded its model build the same way.
        if self.world > 1:
            dist.broadcast(self.flat_params, src=dist.get_global_rank(process_group, 0) if process_group is not None else 0,
                           group=process_group)
        # step() draws noise / timesteps from PER-RANK generators (seed + rank): with one global seed on every rank (the
        # usual way to build identical replicas) the default generators would hand every rank the same t and noise for
        # its different images.  seed=None keeps the reference's behaviour on one process (global generators, :99-102).
        self._gen_cpu = self._gen_dev = None
        if seed is not None or self.world > 1:
            base = 0 if seed is None else int(seed)
            self._gen_cpu = torch.Generator().manual_seed(base + self.rank)
            self._gen_dev = torch.Generator(device=dev).manual_seed(base + self.rank)

    # ---- torch.optim.Adam-compatible views of the optimizer state (for checkpoints, train_ddpm.py:55-61) ----
    def export_optimizer_state(self, optimizer):
        """Make ``optimizer.state`` point at this trainer's moment buffers so ``optimizer.state_dict()`` saves them."""
        params = dict(self.model.named_parameters())
        for name, (off, n) in self.slices.items():
            p = params[name]
            optimizer.state[p] = {"step": torch.tensor(float(self.step_count)),
                                  "exp_avg": self.exp_avg[off:off + n].view(p.shape),
                                  "exp_avg_sq": self.exp_avg_sq[off:off + n].view(p.shape)}

    def import_optimizer_state(self, optimizer):
        """Resume (train_ddpm.py:63-68,81-84: load_checkpoint fills the optimizer before train()): copy ``exp_avg``,
        ``exp_avg_sq`` and ``step`` of a torch.optim.Adam whose state is keyed by this model's parameters into the flat
        moment buffers.  Returns the number of parameters restored (0 when the optimizer has no state yet)."""
        params = dict(self.model.named_parameters())
        restored, steps = 0, set()
        for name, (off, n) in self.slices.items():
            st = optimizer.state.get(params[name])
            if not st or "exp_avg" not in st:
                continue
            self.exp_avg[off:off + n].copy_(st["exp_avg"].reshape(-1).to(self.exp_avg.device, torch.float32))
            self.exp_avg_sq[off:off + n].copy_(st["exp_avg_sq"].reshape(-1).to(self.exp_avg.device, torch.float32))
            steps.add(int(float(st["step"])))
            restored += 1
        if restored:
            if restored != len(self.slices) or len(steps) != 1:
                raise RuntimeError("optimizer state covers only part of the model or has mixed step counts; cannot resume")
            self.step_count = steps.pop()
        return restored

    def _bind(self, B, H, W):
        if self._bound == (B, H, W):
            return
        L, dev = lib(), self.flat_params.device
        if self._plan is None:
            params = {s: self.flat_params[o:o + n] for s, (o, n) in self.slices.items()}     # in self.names order
            grads = {s: self.flat_grads[o:o + n] for s, (o, n) in self.slices.items()}
            c_names, pp, _ = c_tensor_args(params, dev, "DenoisingTrainer")
            _, gp, _ = c_tensor_args(grads, dev, "DenoisingTrainer")
            cfg = self.model._config_struct()
            self._plan = PlanHandle(L.wc_unet_train_create, L.wc_unet_train_destroy, C.byref(cfg), len(self.names), c_names,
                                    pp, gp, keep=(self.flat_params, self.flat_grads))
        handle = self._plan.handle
        ws = self._plan.workspace((B, H, W), lambda: L.wc_unet_train_workspace_bytes(handle, B, H, W), dev)
        check(L.wc_unet_train_bind(handle, B, H, W, ptr(ws), ws.numel(), stream_ptr()))
        self._bound = (B, H, W)
        # ---- gradient buckets: contiguous slices of the flat buffer, closed when the backward plan is done with them
        n_ops = L.wc_unet_train_num_backward_ops(handle)
        ready = [L.wc_unet_train_grad_ready_op(handle, s.encode()) for s in self.names]
        if min(ready) < 0:
            raise RuntimeError("internal: a parameter has no gradient producer: " + self.names[ready.index(min(ready))])
        self._buckets = make_buckets(self.names, self.slices, self.groups, ready, n_ops, self.used, self.bucket_bytes)
        self._n_bwd_ops = n_ops

    @property
    def flops_per_step(self):
        L, plan = lib(), self._plan
        return float(L.wc_unet_train_flops(plan.handle, 0) + L.wc_unet_train_flops(plan.handle, 1)) if plan else 0.0

    def forward_backward(self, noisy, t, target, pred_out=None):
        """loss (device scalar) and all gradients for pred = model(noisy, t), loss = MSE(pred, target)."""
        _lib.require_cuda(noisy, target)
        noisy, target = noisy.contiguous().float(), target.contiguous().float()
        B, _, H, W = noisy.shape
        t = torch.as_tensor(t).long().to(noisy.device).reshape(-1).contiguous()
        if t.numel() != B:
            raise RuntimeError("training needs one timestep per sample")
        self._bind(B, H, W)
        L, st, handle = lib(), stream_ptr(), self._plan.handle
        check(L.wc_unet_train_forward(handle, ptr(noisy), ptr(t), ptr(target), ptr(pred_out), ptr(self.loss), 1.0, 1, st))
        backward_with_buckets(lambda a, b: check(L.wc_unet_train_backward(handle, a, b, st)), self._n_bwd_ops,
                              self.flat_grads, self._buckets, self.world, self.group)
        self._keep = (noisy, t, target, pred_out)
        return self.loss

    def optimizer_step(self):
        self.step_count += 1
        self.model._weights_epoch += 1      # the inference plan re-packs its weights on its next call
        check(lib().wc_adam_step(ptr(self.flat_params), ptr(self.flat_grads), ptr(self.exp_avg), ptr(self.exp_avg_sq),
                                 self.used, self.lr, self.betas[0], self.betas[1], self.eps, self.step_count,
                                 1.0 / self.world, stream_ptr()))

    def step(self, images, noise=None, t=None):
        """One reference training step (train_ddpm.py:95-114); returns the loss as a device scalar tensor."""
        images = images.float().to(self.flat_params.device)
        if noise is None:
            noise = torch.randn(images.shape, device=images.device, generator=self._gen_dev)               # :99
        if t is None:                                                               # :102 (CPU generator, then H2D)
            t = torch.randint(0, self.scheduler.num_timesteps, (images.shape[0],), generator=self._gen_cpu)
        t = torch.as_tensor(t).to(images.device)
        noisy = self.scheduler.add_noise(images, noise, t)                          # :105
        loss = self.forward_backward(noisy, t, noise)                               # :106-109
        self.optimizer_step()                                                       # :113
        return loss


def fused_step_supported(criterion, optimizer) -> bool:
    """True when (criterion, optimizer) is exactly what the fused step computes: mean-reduced nn.MSELoss and
    torch.optim.Adam without weight decay, amsgrad or maximize (subclasses may change either, so the types must match)."""
    if type(criterion) is not torch.nn.MSELoss or criterion.reduction != "mean":
        return False
    if type(optimizer) is not torch.optim.Adam:
        return False
    return all(not g.get("weight_decay", 0) and not g.get("amsgrad", False) and not g.get("maximize", False)
               for g in optimizer.param_groups)


def _train_generic(dataloader, model, optimizer, criterion, scheduler, epochs, log_interval, on_log, on_epoch_end, seed,
                   process_group):
    """The reference's step body (train_ddpm.py:95-114) verbatim on the differentiable Unet, with noise and t drawn as
    DenoisingTrainer.step draws them."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(process_group) > 1:
        raise RuntimeError("train(): data parallelism runs on the fused step only (nn.MSELoss() + torch.optim.Adam); "
                           f"got {type(criterion).__name__} + {type(optimizer).__name__}")
    dev = next(model.parameters()).device
    if dev.type != "cuda":
        raise RuntimeError("move the model to the GPU before training")
    gen_cpu = gen_dev = None
    if seed is not None:
        gen_cpu = torch.Generator().manual_seed(int(seed))
        gen_dev = torch.Generator(device=dev).manual_seed(int(seed))
    was_differentiable = model.differentiable
    model.differentiable = True
    losses = []
    try:
        for epoch_idx in range(1, epochs + 1):
            interval = 0.0
            for batch_idx, images in enumerate(dataloader):
                optimizer.zero_grad()
                images = images.float().to(dev)
                noise = torch.randn(images.shape, device=dev, generator=gen_dev)                # :99
                t = torch.randint(0, scheduler.num_timesteps, (images.shape[0],), generator=gen_cpu).to(dev)   # :102
                noisy = scheduler.add_noise(images, noise, t)                                   # :105
                noise_pred = model(noisy, t)                                                    # :106-109
                loss = criterion(noise_pred, noise)
                loss.backward()
                optimizer.step()                                                                # :113
                interval += float(loss)
                losses.append(float(loss))
                if (batch_idx + 1) % log_interval == 0:
                    if on_log is not None:
                        on_log(epoch_idx, batch_idx + 1, interval / log_interval)
                    interval = 0.0
            if on_epoch_end is not None:
                on_epoch_end(epoch_idx)
    finally:
        model.differentiable = was_differentiable
    return losses


def train(dataloader, model: Unet, optimizer, criterion, scheduler, epochs=1, log_interval=10, on_log=None, on_epoch_end=None,
          seed=None, process_group=None):
    """Drop-in for the reference's ``train`` (train_ddpm.py:71-133): same arguments, same return value (the per-step
    losses).  For ``nn.MSELoss()`` with ``torch.optim.Adam`` (no weight decay / amsgrad / maximize; the reference's pair,
    :151-152) the step is the fused DenoisingTrainer step: the Adam hyper-parameters are read from ``optimizer``, and an
    ``optimizer`` that already carries state (the reference's load_checkpoint, :63-68,81-84) has its moments and step count
    imported, so Adam continues instead of restarting.  ``optimizer.state`` is re-pointed at the live moment buffers before
    every ``on_log`` and ``on_epoch_end(epoch)`` call (the reference's per-epoch save_checkpoint, :135-141), so
    ``optimizer.state_dict()`` taken inside those hooks is a valid checkpoint.  Any other criterion or optimizer runs the
    reference's step body on the differentiable Unet (one GPU only), where ``optimizer.state`` is the real state.  wandb /
    tqdm / file I/O of the reference are host-side plumbing left to the two hooks."""
    if not fused_step_supported(criterion, optimizer):
        return _train_generic(dataloader, model, optimizer, criterion, scheduler, epochs, log_interval, on_log,
                              on_epoch_end, seed, process_group)
    g = optimizer.param_groups[0]
    trainer = DenoisingTrainer(model, scheduler, lr=g["lr"], betas=g["betas"], eps=g["eps"], seed=seed,
                               process_group=process_group)
    trainer.import_optimizer_state(optimizer)
    losses = []
    for epoch_idx in range(1, epochs + 1):
        interval = 0.0
        for batch_idx, images in enumerate(dataloader):
            loss = trainer.step(images)
            interval += float(loss)          # the reference also reads loss.item() every step (:116)
            losses.append(float(loss))
            if (batch_idx + 1) % log_interval == 0:
                if on_log is not None:
                    trainer.export_optimizer_state(optimizer)
                    on_log(epoch_idx, batch_idx + 1, interval / log_interval)
                interval = 0.0
        trainer.export_optimizer_state(optimizer)
        if on_epoch_end is not None:
            on_epoch_end(epoch_idx)
    trainer.export_optimizer_state(optimizer)
    return losses
