"""CUDA-graph replay of `MipNerf.forward` for a fixed batch shape.

A 4096-ray forward is two kernel launches (~0.5 ms each on a B200) plus a 12 KB constant upload; the host side of
one call (ctypes marshalling, output allocation, argument checks) costs ~85 us, and at 512 rays per GPU (the
4096-ray batch split over 8 GPUs) the launch path is as long as the kernels.  `GraphedForward` captures ONE forward
— and, for a ray-sharded batch, the NCCL all-gather of the rendered pixels that follows it (the reference's only
inference-time collective is implicit in its single-GPU loop; its training collective is DDP's, train.py:60) — into
a CUDA graph on static buffers and replays it: one `cudaGraphLaunch` per step.  `GraphedTrainStep` does the same for
a whole training step (DESIGN.md §8c).

The rays live in a `RayStaging` device buffer (one H2D copy per step refreshes them), the outputs in the tensors
the captured forward returned; both keep their addresses for the life of the object.
"""
from __future__ import annotations

import os
from typing import Optional

import torch

from .rays import Rays, RayStaging


class GraphedForward:
    def __init__(self, model, staging: RayStaging, white_bkgd: bool = True, device=None, world: int = 1,
                 group=None, gather: str = "fine_rgb", warmup: int = 3):
        """`staging`: this rank's rays (its shard of the global batch).  world > 1: every replay ends with one
        all_gather_into_tensor of this rank's fine RGB ([B,3]) or of all pixels (`gather='pixels'`: rgb, distance,
        acc of both levels, 10 floats per ray) into `self.gathered`."""
        self.model, self.staging, self.white = model, staging, bool(white_bkgd)
        self.device = torch.device(device) if device is not None else next(model.parameters()).device
        self.world, self.group, self.gather = int(world), group, gather
        b = staging.num_rays
        self.rays: Rays = staging.to(self.device)            # static input buffer (views of one allocation)
        self.gathered: Optional[torch.Tensor] = None
        if self.world > 1:
            width = 3 if gather == "fine_rgb" else 10
            self.gathered = torch.empty(self.world * b * width, device=self.device)
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(side), torch.no_grad():
            for _ in range(max(1, warmup)):                   # kernels loaded, NCCL communicator built, caches warm
                self._run()
        torch.cuda.current_stream(self.device).wait_stream(side)
        torch.cuda.synchronize(self.device)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph), torch.no_grad():
            self.ret = self._run()

    def _run(self):
        ret = self.model(self.rays, False, self.white)
        if self.world > 1:
            import torch.distributed as dist
            src = ret[-1][0] if self.gather == "fine_rgb" else ret.pixels
            dist.all_gather_into_tensor(self.gathered, src.reshape(-1), group=self.group)
        return ret

    def load(self, non_blocking: bool = True) -> None:
        """One H2D copy of the staging buffer's current host contents into the graph's input."""
        self.staging.to(self.device, non_blocking=non_blocking)

    def replay(self):
        """One graph launch on the current stream; returns the (static) LevelOutputs of the captured forward."""
        self.graph.replay()
        return self.ret

    def __call__(self, rays: Optional[Rays] = None):
        if rays is not None:
            self.staging.fill(rays)
            self.load()
        return self.replay()


class GraphedTrainStep:
    """One whole training step -- batch sampling, fused forward + backward, loss, the DDP all-reduce (world > 1),
    Adam with the MipLRDecay schedule, counter advance and loss logging -- captured into ONE CUDA graph with every piece
    of step state on the device:

    * `rng_state` int64 [2]: the Philox (seed, offset) that the sampler and the level kernels read when they run;
      the step ends with offset += 1, as `MipNerf.next_rng` does per eager step;
    * `step` int64 [1]: Adam's step count; the update reads lr / bc1 and sqrt(bc2) from tables indexed by it
      (`train.adam_tables`), so it equals FusedAdam stepped with MipLRDecay bit for bit;
    * `ring` [ring_len, 2]: (loss, fine PSNR) of step s in row s % ring_len.

    `replay(k)` launches k steps without a host synchronisation.  `sync()` hands the device state back to the host
    objects (optimiser step counts, `model.rng_offset`, the scheduler) so that an eager step, a checkpoint or a
    render sees a consistent model, and returns the logged rows.  BF16 / FP16 fused step only.

    Pixel ids come from the batch sampler of `bank` (`DeviceRayBank.sample_philox`, ray_base 0).  With world > 1 each
    rank samples its own `batch_size` rays: give every rank its own `model.rng_seed` (fit() uses seed + rank)."""

    def __init__(self, model, optimizer, scheduler, bank, batch_size: int, *, randomized: bool = True,
                 white_bkgd: bool = True, coarse_loss_mult: float = 0.1, dist_mult: float = 0.01,
                 disable_multiscale_loss: bool = False, num_steps: Optional[int] = None, ring_len: int = 1024,
                 world: int = 1, group=None, warmup: int = 2):
        import numpy as np
        from .mip_nerf import _Workspace
        from .train import _grads_ready, _level_multipliers, adam_tables
        if model.precision not in ("bf16", "fp16"):
            raise NotImplementedError(f"GraphedTrainStep: the fused BF16 / FP16 step only (precision={model.precision!r})")
        if os.environ.get("MIPNERF_B200_TRAIN_FUSED", "1")[:1] == "0":
            raise NotImplementedError("GraphedTrainStep: MIPNERF_B200_TRAIN_FUSED=0 selects the unfused step")
        if len(optimizer.param_groups) != 1:
            raise ValueError("GraphedTrainStep: one parameter group (the MLP's 24 tensors)")
        self.model, self.opt, self.sched, self.bank = model, optimizer, scheduler, bank
        self.batch_size, self.randomized, self.white = int(batch_size), bool(randomized), bool(white_bkgd)
        self.coarse_loss_mult, self.dist_mult = float(coarse_loss_mult), float(dist_mult)
        self.disable_multiscale_loss = bool(disable_multiscale_loss)
        self.world, self.group = int(world), group
        self.device = dev = next(model.parameters()).device
        self.params = _grads_ready(model)
        group0 = optimizer.param_groups[0]
        if {id(p) for p in group0["params"]} != {id(p) for p in self.params}:
            raise ValueError("GraphedTrainStep: the optimiser must hold exactly the model's MLP parameters")
        for p in self.params:
            st = optimizer.state[p]
            if not st:
                st["step"] = 0
                st["exp_avg"] = torch.zeros_like(p)
                st["exp_avg_sq"] = torch.zeros_like(p)
        steps = {optimizer._step_count(optimizer.state[p]) for p in self.params}
        if len(steps) != 1:
            raise ValueError("GraphedTrainStep: parameters at different Adam steps")
        start = steps.pop()
        self.num_steps = int(num_steps if num_steps is not None else max(scheduler.max_steps, start + 1))
        step_size, bc2_sqrt = adam_tables(self.num_steps, group0["betas"], scheduler.lr_init, scheduler.lr_final,
                                          scheduler.max_steps, scheduler.lr_delay_steps, scheduler.lr_delay_mult)
        self.step_size = torch.from_numpy(step_size).to(dev)
        self.bc2_sqrt = torch.from_numpy(bc2_sqrt).to(dev)
        if model.rng_seed is None:
            model.rng_seed = int(torch.initial_seed()) & 0xFFFFFFFFFFFFFFFF
        self.step = torch.tensor([start], dtype=torch.int64, device=dev)
        self.rng_state = torch.tensor(np.array([model.rng_seed, model.rng_offset], dtype=np.uint64).view(np.int64),
                                      device=dev)
        self.ring_len = int(ring_len)
        self.ring = torch.full((max(self.ring_len, 1), 2), float("nan"), device=dev)
        self._host_step = start          # step count the host knows the device is at after the queued replays
        self._synced_step = start
        levels = model.num_levels
        mse_m, dist_m = _level_multipliers(levels, self.coarse_loss_mult, self.dist_mult)
        self.level_mults = (torch.tensor(mse_m, device=dev), torch.tensor(dist_m, device=dev))
        self.mask_sum = torch.tensor([float(self.batch_size)], device=dev) if self.disable_multiscale_loss else None
        self.batch = bank.sample_philox(self.rng_state, self.batch_size)   # static (Rays, rgb, ids) buffers
        self._adam_args = self._adam_arrays()

        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        snapshot = self._state_tensors()
        saved = [t.clone() for t in snapshot]
        with torch.cuda.stream(side), torch.no_grad():
            for _ in range(max(1, warmup)):   # kernels loaded, workspace and NCCL communicator built; state restored
                self._run()
            for t, s in zip(snapshot, saved):
                t.copy_(s)
            # the forward_backward scratch the graph will write on every replay: held here, so that a later, larger
            # request on a stream with the same handle (torch recycles them) cannot free it under the graph
            self._scratch = _Workspace.get(dev, 0)
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        del saved
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph, stream=side), torch.no_grad():
            self.out = self._run()

    def _state_tensors(self):
        st = [self.opt.state[p] for p in self.params]
        return ([p.data for p in self.params] + [s["exp_avg"] for s in st] + [s["exp_avg_sq"] for s in st] +
                [self.step, self.rng_state, self.ring])

    def _adam_arrays(self):
        import ctypes as C
        n = len(self.params)
        arr = C.c_void_p * n
        st = [self.opt.state[p] for p in self.params]
        return (n, arr(*[p.data_ptr() for p in self.params]), arr(*[p.grad.data_ptr() for p in self.params]),
                arr(*[s["exp_avg"].data_ptr() for s in st]), arr(*[s["exp_avg_sq"].data_ptr() for s in st]),
                (C.c_int64 * n)(*[p.numel() for p in self.params]))

    def _run(self):
        from . import _cabi
        from .nerf_system import calc_psnr
        from .ops import _stream
        from .train import _run, allreduce_grads
        self.bank.sample_philox(self.rng_state, self.batch_size, out=self.batch)
        rays, rgb, _ = self.batch
        out = _run(self.model, rays, rgb, self.randomized, self.white, self.coarse_loss_mult, self.dist_mult,
                   self.disable_multiscale_loss, None, None, [p.grad for p in self.params], False, self.mask_sum, None,
                   rng_state=self.rng_state, level_mults=self.level_mults)
        psnr = calc_psnr(out["ret"][-1][0], rgb)
        if self.world > 1:
            allreduce_grads(self.params, self.group)
        g = self.opt.param_groups[0]
        lib = _cabi.lib()
        n, ps, gs, ms, vs, sizes = self._adam_args
        _cabi.check(lib.mipnerf_b200_adam_step_multi_table(
            n, ps, gs, ms, vs, sizes, self.step_size.data_ptr(), self.bc2_sqrt.data_ptr(), self.step_size.numel(),
            self.step.data_ptr(), float(g["betas"][0]), float(g["betas"][1]), float(g["eps"]),
            float(g.get("grad_scale", 1.0)), _stream(self.device)), "GraphedTrainStep adam")
        _cabi.check(lib.mipnerf_b200_train_step_advance(
            self.step.data_ptr(), self.rng_state.data_ptr(), out["loss"].data_ptr(), psnr.data_ptr(),
            self.ring.data_ptr(), self.ring_len, _stream(self.device)), "GraphedTrainStep advance")
        out["psnr"] = psnr
        return out

    def replay(self, k: int = 1) -> None:
        """k training steps, one graph launch each, on the current stream; no host synchronisation."""
        if self._host_step + k > self.num_steps:
            raise ValueError(f"GraphedTrainStep: step {self._host_step + k} is past the {self.num_steps} steps "
                             "the Adam tables cover (num_steps)")
        for _ in range(k):
            self.graph.replay()
        self._host_step += k

    def sync(self):
        """Wait for the queued steps; write the step count into the optimiser state, the Philox offset into
        `model.rng_offset` and the schedule into the scheduler; return [(step, loss, psnr)] of the steps since the
        last sync that the ring still holds."""
        ring = self.ring.cpu()
        step = int(self.step.item())
        offset = int(self.rng_state[1].item()) & 0xFFFFFFFFFFFFFFFF
        for p in self.params:
            self.opt.state[p]["step"] = step
            torch.autograd.graph.increment_version(p)   # written in place by the graph: keep the weight caches honest
        self.model.rng_offset = offset
        self.sched.last_epoch = step
        lrs = self.sched.get_lr()
        for g, lr in zip(self.opt.param_groups, lrs):
            g["lr"] = lr
        self.sched._last_lr = list(lrs)
        first = max(self._synced_step, step - self.ring_len) if self.ring_len > 0 else step
        rows = [(s + 1, float(ring[s % self.ring_len, 0]), float(ring[s % self.ring_len, 1])) for s in range(first, step)]
        self._synced_step = self._host_step = step
        return rows
