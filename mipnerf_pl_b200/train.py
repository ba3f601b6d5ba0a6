"""Training step of `MipNeRFSystem` (models/nerf_system.py:70-76, 95-121) on the library's backward
kernels (SURVEY.md §8f N2).  `MipNerf.precision` selects the arithmetic of the step: 'fp32' = every GEMM in fp32
FFMA (the parity mode, gradients match the reference's autograd); 'bf16' / 'fp16' = forward and dgrad GEMMs on
tcgen05 with 16-bit operands and fp32 accumulation, wgrad / heads / rendering in fp32.

* `fused_loss(...)`       the reference's training loss as one differentiable scalar: forward + backward run
                          inside `mipnerf_b200_forward_backward`; `loss.backward()` only hands the stored
                          gradients to autograd, so Lightning / any torch optimiser drives it unchanged.
* `forward_backward(...)` the same without autograd: gradients land in `param.grad` directly.
* `FusedAdam`             torch.optim.Adam semantics, update done by `mipnerf_b200_adam_step`.
* `MipLRDecay`, `mip_lr`  utils/lr_schedule.py:51-60 (log-linear decay with the delayed warm-up).
* `allreduce_grads`       DDP's gradient all-reduce over the ray shards: ONE collective on a flat buffer.
* `adam_tables`           the per-step (lr/bc1, sqrt(bc2)) of FusedAdam + MipLRDecay for the captured training step
                          (graph.GraphedTrainStep), computed with the host math FusedAdam hands the library.

Gradients do not flow into the fenceposts (stop_resample_grad=True, the reference default); a model built
with stop_resample_grad=False is refused rather than silently trained with different gradients.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Dict, Iterable, List, Optional, Sequence

import torch

from . import _cabi
from .mip_nerf import MipNerf, _Workspace
from .ops import _dev, _f32, _ptr, _stream, draw_density_normal, draw_t_rand, draw_u_jitter
from .rays import Rays


def mip_lr(step: int, lr_init: float, lr_final: float, max_steps: int, lr_delay_steps: int = 0,
           lr_delay_mult: float = 1.0) -> float:
    """utils/lr_schedule.py:51-60."""
    if lr_delay_steps > 0:
        delay_rate = lr_delay_mult + (1 - lr_delay_mult) * math.sin(
            0.5 * math.pi * min(max(step / lr_delay_steps, 0.0), 1.0))
    else:
        delay_rate = 1.0
    t = min(max(step / max_steps, 0.0), 1.0)
    return delay_rate * math.exp(math.log(lr_init) * (1 - t) + math.log(lr_final) * t)


class MipLRDecay(torch.optim.lr_scheduler.LRScheduler):
    """utils/lr_schedule.py:5-60: same constructor, one param group, stepped every optimiser step."""

    def __init__(self, optimizer, lr_init: float, lr_final: float, max_steps: int, lr_delay_steps: int,
                 lr_delay_mult: float):
        self.lr_init, self.lr_final, self.max_steps = lr_init, lr_final, max_steps
        self.lr_delay_steps, self.lr_delay_mult = lr_delay_steps, lr_delay_mult
        super().__init__(optimizer)

    def get_lr(self):
        return [mip_lr(self.last_epoch, self.lr_init, self.lr_final, self.max_steps, self.lr_delay_steps,
                       self.lr_delay_mult)]


class FusedAdam(torch.optim.Optimizer):
    """torch.optim.Adam(params, lr) (models/nerf_system.py:71-72) with the update done on the device by one
    library kernel per tensor.  `grad_scale` multiplies the gradient as it is read (1/world_size after a
    sum all-reduce)."""

    def __init__(self, params, lr: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8, grad_scale: float = 1.0):
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, grad_scale=grad_scale))

    @staticmethod
    def _step_count(st) -> int:
        """Steps taken so far as a Python int: a state loaded from a torch.optim.Adam checkpoint (what the reference's
        Lightning `trainer.fit(ckpt_path=...)` restores) keeps `step` as a float32 tensor."""
        step = st["step"]
        return step if isinstance(step, int) else int(float(step))

    def _step_group(self, lib, group, b1: float, b2: float, grad_scale: float) -> bool:
        """One launch for the whole group (`mipnerf_b200_adam_step_multi`) when its tensors sit on one CUDA device
        and share a step count — the normal case; otherwise the caller falls back to one launch per tensor."""
        ps = [p for p in group["params"] if p.grad is not None]
        if not ps or any(p.dtype != torch.float32 or not p.is_contiguous() or not p.grad.is_contiguous() or
                         p.device != ps[0].device or not p.is_cuda for p in ps):
            return False
        for p in ps:
            st = self.state[p]
            if not st:
                st["step"] = 0
                st["exp_avg"] = torch.zeros_like(p)
                st["exp_avg_sq"] = torch.zeros_like(p)
        steps = {self._step_count(self.state[p]) for p in ps}
        if len(steps) != 1:
            return False
        step = steps.pop() + 1
        n = len(ps)
        arr = C.c_void_p * n
        dev = _dev(ps[0])
        with torch.cuda.device(dev):
            _cabi.check(lib.mipnerf_b200_adam_step_multi(
                n, arr(*[p.data_ptr() for p in ps]), arr(*[p.grad.data_ptr() for p in ps]),
                arr(*[self.state[p]["exp_avg"].data_ptr() for p in ps]),
                arr(*[self.state[p]["exp_avg_sq"].data_ptr() for p in ps]),
                (C.c_int64 * n)(*[p.numel() for p in ps]), float(group["lr"]), b1, b2, float(group["eps"]), step,
                grad_scale, _stream(dev)), "FusedAdam.step")
        for p in ps:
            self.state[p]["step"] = step
            torch.autograd.graph.increment_version(p)  # written in place by the library: keep the packed-weight
            #                                            caches (keyed on _version) honest
        return True

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        lib = _cabi.lib()
        for group in self.param_groups:
            b1, b2 = group["betas"]
            grad_scale = float(group.get("grad_scale", 1.0))   # absent after loading a torch.optim.Adam state_dict
            if self._step_group(lib, group, float(b1), float(b2), grad_scale):
                continue
            for p in group["params"]:
                if p.grad is None:
                    continue
                dev = _dev(p)
                if p.dtype != torch.float32 or not p.is_contiguous() or not p.grad.is_contiguous():
                    raise RuntimeError("FusedAdam: contiguous fp32 parameters only")
                st = self.state[p]
                if not st:
                    st["step"] = 0
                    st["exp_avg"] = torch.zeros_like(p)
                    st["exp_avg_sq"] = torch.zeros_like(p)
                st["step"] = self._step_count(st) + 1
                with torch.cuda.device(dev):
                    _cabi.check(lib.mipnerf_b200_adam_step(
                        p.data_ptr(), p.grad.data_ptr(), st["exp_avg"].data_ptr(), st["exp_avg_sq"].data_ptr(),
                        p.numel(), float(group["lr"]), float(b1), float(b2), float(group["eps"]), st["step"],
                        grad_scale, _stream(dev)), "FusedAdam.step")
                torch.autograd.graph.increment_version(p)  # written in place by the library: keep the
                #                                            packed-weight caches (keyed on _version) honest
        return loss


def _flat_view(grads) -> Optional[torch.Tensor]:
    """The one contiguous tensor the gradients are consecutive views of, or None."""
    g0 = grads[0]
    if not all(g.is_contiguous() and g.dtype == g0.dtype and g.device == g0.device for g in grads):
        return None
    store = g0.untyped_storage()
    off = g0.storage_offset()
    for g in grads:
        if g.untyped_storage().data_ptr() != store.data_ptr() or g.storage_offset() != off:
            return None
        off += g.numel()
    return torch.empty(0, dtype=g0.dtype, device=g0.device).set_(store, g0.storage_offset(), (off - g0.storage_offset(),))


def allreduce_grads(params: Iterable[torch.Tensor], group=None, average: bool = True) -> None:
    """DDP semantics (train.py:60 of the reference) for the ray-sharded step: one all-reduce of all
    gradients as a flat buffer, then scattered back into `p.grad`."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return
    grads = [p.grad for p in params if p.grad is not None]
    if not grads:
        return
    flat = _flat_view(grads)
    if flat is not None:                    # gradients already live back to back in one buffer (forward_backward)
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
        if average:
            flat /= dist.get_world_size(group)
        return
    flat = torch.cat([g.reshape(-1) for g in grads])
    dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    if average:
        flat /= dist.get_world_size(group)
    off = 0
    for g in grads:
        g.copy_(flat[off:off + g.numel()].view_as(g))
        off += g.numel()


def adam_tables(num_steps: int, betas, lr_init: float, lr_final: float, max_steps: int, lr_delay_steps: int = 0,
                lr_delay_mult: float = 1.0):
    """float32 tables (step_size, bc2_sqrt) of length num_steps + 1: entry t (t >= 1) is what update t of FusedAdam
    stepped with MipLRDecay uses -- lr = mip_lr(t - 1) (the scheduler has stepped t - 1 times), bc1 = 1 - b1^t,
    bc2 = 1 - b2^t in double, then (float)(lr / bc1) and (float)sqrt(bc2) as mipnerf_b200_adam_step_multi rounds
    them.  Entry 0 is unused."""
    import numpy as np
    b1, b2 = float(betas[0]), float(betas[1])
    step_size = np.zeros(num_steps + 1, dtype=np.float32)
    bc2_sqrt = np.ones(num_steps + 1, dtype=np.float32)
    for t in range(1, num_steps + 1):
        lr = mip_lr(t - 1, lr_init, lr_final, max_steps, lr_delay_steps, lr_delay_mult)
        step_size[t] = np.float32(lr / (1.0 - math.pow(b1, float(t))))
        bc2_sqrt[t] = np.float32(math.sqrt(1.0 - math.pow(b2, float(t))))
    return step_size, bc2_sqrt


def _level_multipliers(num_levels: int, coarse_loss_mult: float, dist_mult: float):
    """loss = coarse_loss_mult * (mse_coarse + 0.01 dist_coarse) + mse_fine + 0.01 dist_fine
    (models/nerf_system.py:110-111; every level before the last counts as coarse)."""
    mse = [coarse_loss_mult] * (num_levels - 1) + [1.0]
    dist = [coarse_loss_mult * dist_mult] * (num_levels - 1) + [dist_mult]
    return mse, dist


def _run(model: MipNerf, rays: Rays, rgbs: torch.Tensor, randomized: bool, white_bkgd: bool,
         coarse_loss_mult: float, dist_mult: float, disable_multiscale_loss: bool, t_rand, u_jitter,
         grad_tensors: Sequence[torch.Tensor], accumulate: bool, mask_sum, global_rays, density_normal=None,
         rng_state: Optional[torch.Tensor] = None, level_mults=None):
    """`rng_state` (int64 [2] on the device, read as uint64 seed / offset by the kernels) replaces `model.next_rng()`
    for randomized=True; `level_mults` = (mse, dist) multipliers [levels] already on the device.  Both exist so that
    the call can be captured into a CUDA graph (no host-to-device copy, no host-side state)."""
    if not model.stop_resample_grad:
        raise NotImplementedError("training kernels implement stop_resample_grad=True (the reference default)")
    prec = _cabi.PRECISIONS[model.precision]   # fp32: the parity mode; bf16 / fp16: forward + dgrad GEMMs on tcgen05
    if model.ray_shape != "cone":
        raise NotImplementedError
    dev = _dev(rays.origins)
    b, n, levels = rays.origins.shape[0], model.num_samples, model.num_levels
    cfg = model._config()
    keep = [_f32(rays.origins), _f32(rays.directions), _f32(rays.viewdirs), _f32(rays.radii).reshape(-1),
            _f32(rays.near).reshape(-1), _f32(rays.far).reshape(-1)]
    rs = _cabi.RaysStruct(*[k.data_ptr() for k in keep], b)
    rng = None
    noisy = bool(randomized) and model.density_noise > 0    # models/mip_nerf.py:232-233
    normals = [None] * levels
    if randomized and rng_state is not None:
        pass                            # (seed, offset) read from the device when the kernels run
    elif randomized and t_rand is None and u_jitter is None and density_normal is None:
        rng = model.next_rng()          # uniforms / normals drawn inside the kernels (Philox), as every training step does
    elif randomized:
        t_rand = _f32(t_rand) if t_rand is not None else draw_t_rand(b, n, dev)
        u_jitter = _f32(u_jitter) if u_jitter is not None else draw_u_jitter(b, n + 1, dev)
        if noisy:
            given = list(density_normal) if density_normal is not None else [None] * levels
            if len(given) != levels:
                raise ValueError(f"density_normal: expected {levels} tensors (one per level)")
            normals = [_f32(x).reshape(b, n) if x is not None else draw_density_normal(b, n, dev) for x in given]
    else:
        t_rand = u_jitter = None
    target = _f32(rgbs[..., :3]).reshape(b, 3)
    mask = None if disable_multiscale_loss else _f32(rays.lossmult).reshape(b)
    if mask_sum is None:
        mask_sum = mask.sum() if mask is not None else torch.tensor(float(b), device=dev)
    mask_sum = _f32(mask_sum).reshape(1)
    global_rays = int(global_rays) if global_rays is not None else b
    mse_m, dist_m = _level_multipliers(levels, coarse_loss_mult, dist_mult)
    mse_arr, dist_arr = (C.c_float * levels)(*mse_m), (C.c_float * levels)(*dist_m)
    sqerr = torch.empty(levels, b, device=dev)
    dl = torch.empty(levels, b, device=dev)
    loss = _cabi.Loss(target.data_ptr(), _ptr(mask), mask_sum.data_ptr(), 1.0 / max(global_rays, 1), mse_arr, dist_arr,
                      sqerr.data_ptr(), dl.data_ptr())
    ws, wkeep = model.mlp._weights_struct(cfg, _cabi.FP32, dev)
    lins = model.mlp.linears()
    assert len(grad_tensors) == 2 * len(lins)
    garr = (_cabi.LinearGrad * len(lins))()
    for i in range(len(lins)):
        garr[i] = _cabi.LinearGrad(grad_tensors[2 * i].data_ptr(), grad_tensors[2 * i + 1].data_ptr())
    outs = (_cabi.LevelOut * levels)()
    ret = []
    for lvl in range(levels):
        comp, dist, acc = torch.empty(b, 3, device=dev), torch.empty(b, device=dev), torch.empty(b, device=dev)
        w, t = torch.empty(b, n, device=dev), torch.empty(b, n + 1, device=dev)
        outs[lvl] = _cabi.LevelOut(comp.data_ptr(), dist.data_ptr(), acc.data_ptr(), w.data_ptr(), t.data_ptr(), None,
                                   _ptr(normals[lvl]))
        ret.append((comp, dist, acc, w, t))
    lib = _cabi.lib()
    nbytes = lib.mipnerf_b200_train_workspace_bytes(C.byref(cfg), b)
    scratch = _Workspace.get(dev, nbytes)
    tail = (int(bool(white_bkgd)), prec, C.byref(loss), outs, garr, len(lins), int(bool(accumulate)),
            scratch.data_ptr() if nbytes else None, scratch.numel() if nbytes else 0, _stream(dev))
    with torch.cuda.device(dev):
        if randomized and rng_state is not None:
            rc = lib.mipnerf_b200_forward_backward_rng_state(C.byref(cfg), C.byref(ws), C.byref(rs), rng_state.data_ptr(),
                                                             *tail)
        elif rng is not None:
            rc = lib.mipnerf_b200_forward_backward_rng(C.byref(cfg), C.byref(ws), C.byref(rs), C.byref(rng), *tail)
        else:
            rc = lib.mipnerf_b200_forward_backward(C.byref(cfg), C.byref(ws), C.byref(rs), int(bool(randomized)),
                                                   _ptr(t_rand), _ptr(u_jitter), *tail)
        _cabi.check(rc, "forward_backward")
    if level_mults is None:
        level_mults = (torch.tensor(mse_m, device=dev), torch.tensor(dist_m, device=dev))
    mse, distl, total = _assemble_loss(sqerr, dl, mask_sum, global_rays, *level_mults)
    return {"loss": total, "mse": mse, "distloss": distl, "ret": ret}


def _assemble_loss(sqerr, dl, mask_sum, global_rays: int, mse_mult: torch.Tensor, dist_mult: torch.Tensor):
    """(mse [levels], distloss [levels], loss) from the per-ray terms the step leaves behind; device ops only."""
    mse = sqerr.sum(dim=1) / mask_sum                      # [levels]   (models/nerf_system.py:104-105)
    distl = dl.sum(dim=1) / max(global_rays, 1)            # [levels]   (:106)
    total = (mse * mse_mult + distl * dist_mult).sum()
    return mse, distl, total


def _param_list(model: MipNerf) -> List[torch.nn.Parameter]:
    return [p for lin in model.mlp.linears() for p in (lin.weight, lin.bias)]


def forward_backward(model: MipNerf, rays: Rays, rgbs: torch.Tensor, randomized: bool, white_bkgd: bool, *,
                     coarse_loss_mult: float = 0.1, dist_mult: float = 0.01, disable_multiscale_loss: bool = False,
                     t_rand=None, u_jitter=None, density_normal=None, accumulate: bool = False, mask_sum=None,
                     global_rays: Optional[int] = None) -> Dict[str, object]:
    """Forward + backward of the training loss; gradients are written (or added, with `accumulate`)
    into `param.grad`.  For a ray shard of a larger batch pass the GLOBAL `mask_sum` / `global_rays`;
    shard gradients then sum to the full-batch gradient."""
    params = _grads_ready(model)
    return _run(model, rays, rgbs, randomized, white_bkgd, coarse_loss_mult, dist_mult, disable_multiscale_loss,
                t_rand, u_jitter, [p.grad for p in params], accumulate, mask_sum, global_rays, density_normal)


def _grads_ready(model: MipNerf) -> List[torch.nn.Parameter]:
    """The MLP's parameters, each with a contiguous `.grad` (carved from one flat buffer on first use)."""
    params = _param_list(model)
    if all(p.grad is None for p in params) and len({(p.device, p.dtype) for p in params}) == 1:
        # first step: carve every .grad out of ONE flat buffer, so that the data-parallel all-reduce
        # (`allreduce_grads`) is a single NCCL call on it with no concatenate / scatter copies
        flat = torch.zeros(sum(p.numel() for p in params), device=params[0].device, dtype=params[0].dtype)
        off = 0
        for p in params:
            p.grad = flat[off:off + p.numel()].view_as(p)
            off += p.numel()
    for p in params:
        if p.grad is None:
            p.grad = torch.zeros_like(p)
        elif not p.grad.is_contiguous():
            p.grad = p.grad.contiguous()
    return params


class _FusedLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, model, rays, rgbs, randomized, white_bkgd, kwargs, holder, *params):
        grads = [torch.empty_like(p) for p in params]
        out = _run(model, rays, rgbs, randomized, white_bkgd, kwargs["coarse_loss_mult"], kwargs["dist_mult"],
                   kwargs["disable_multiscale_loss"], kwargs.get("t_rand"), kwargs.get("u_jitter"), grads, False,
                   kwargs.get("mask_sum"), kwargs.get("global_rays"), kwargs.get("density_normal"))
        holder.update(out)
        ctx.grads = grads
        return out["loss"].clone()

    @staticmethod
    def backward(ctx, grad_out):
        return (None,) * 7 + tuple(g * grad_out for g in ctx.grads)


def fused_loss(model: MipNerf, rays: Rays, rgbs: torch.Tensor, randomized: bool, white_bkgd: bool, *,
               coarse_loss_mult: float = 0.1, dist_mult: float = 0.01, disable_multiscale_loss: bool = False,
               **kw):
    """(loss, info): `loss` is a scalar with a grad_fn over the 24 MLP tensors, numerically the loss of
    models/nerf_system.py:95-111; info holds 'mse', 'distloss' ([levels]) and 'ret' (the forward 5-tuples)."""
    holder: Dict[str, object] = {}
    kwargs = dict(coarse_loss_mult=coarse_loss_mult, dist_mult=dist_mult,
                  disable_multiscale_loss=disable_multiscale_loss, **kw)
    loss = _FusedLoss.apply(model, rays, rgbs, randomized, white_bkgd, kwargs, holder, *_param_list(model))
    return loss, holder
