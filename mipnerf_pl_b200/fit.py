"""Train a scene on the device: the reference's `train.py` (a Lightning `Trainer.fit`) without Lightning.

    python -m mipnerf_pl_b200.fit --data_path DATA --out_dir OUT --dataset_name blender [--config lego.yaml] \
        [key value ...]

* the configuration is a YAML file in the layout of the reference's `configs/lego.yaml` (nested sections) read into
  the flat dotted dict `default_hparams()` returns, then `key value` overrides (`optimizer.max_steps 2000`);
* every step is one replay of `GraphedTrainStep` (batch sampling, fused BF16 / FP16 forward + backward, loss,
  DDP all-reduce, Adam + MipLRDecay, all on the device); the host wakes up once per `val.check_interval` steps;
* validation renders the first `val.sample_num` images of the val split (`render_image` + `eval_errors`);
* `out_dir/ckpt/<exp_name>/last.ckpt` plus the best two by `val/psnr` (`epoch=0-step=<n>.ckpt`), in the layout
  `MipNeRFSystem.load_from_checkpoint` reads, with the optimiser, scheduler and RNG state for
  `checkpoint.resume_path`;
* under torchrun with `num_gpus > 1` every rank samples its own `train.batch_size` rays (Philox seed = seed + rank)
  and the step all-reduces the gradients, as Lightning's DDP does.  Rank 0 validates and writes checkpoints.
"""
from __future__ import annotations

import argparse
import ast
import os
import random
import sys
from typing import Callable, Dict, List, Optional, Sequence

import numpy as np
import torch

from .nerf_system import MipNeRFSystem, default_hparams

DATASETS = ("blender", "multi_blender")


# ---------------------------------------------------------------------------------------------------------------------
# configuration
# ---------------------------------------------------------------------------------------------------------------------
def parse_scalar(text: str):
    """A YAML / command-line scalar: quoted string, None / True / False, int, float, else the bare string
    (so `append_identity: Ture` stays the string 'Ture', as the reference reads it)."""
    t = text.strip()
    if len(t) >= 2 and t[0] == t[-1] and t[0] in "'\"":
        return t[1:-1]
    if t in ("None", "null", "~", ""):
        return None
    if t in ("True", "true"):
        return True
    if t in ("False", "false"):
        return False
    try:
        return int(t)
    except ValueError:
        pass
    try:
        return float(t)
    except ValueError:
        pass
    try:
        v = ast.literal_eval(t)
        return tuple(v) if isinstance(v, list) else v
    except (ValueError, SyntaxError):
        return t


def _strip_comment(line: str) -> str:
    quote = None
    for i, ch in enumerate(line):
        if quote:
            if ch == quote:
                quote = None
        elif ch in "'\"":
            quote = ch
        elif ch == "#" and (i == 0 or line[i - 1] in " \t"):
            return line[:i]
    return line


def read_config(path: str) -> Dict[str, object]:
    """The nested `key: value` sections of a config file as one flat dotted dict ({'train.batch_size': 3072, ...}).
    Block mappings with space indentation and scalar values: the layout of the reference's configs.  A key with
    nothing after the colon and no deeper-indented lines below it is None (YAML's null); every line of a section
    sits at the same indentation, deeper than its header."""
    flat: Dict[str, object] = {}
    stack: List[list] = []           # open sections: [indent, dotted prefix, indent of their lines or None]

    def close(section):
        if section[2] is None:       # `key:` with nothing below it
            flat[section[1][:-1]] = None

    with open(path) as fp:
        for lineno, raw in enumerate(fp, 1):
            line = _strip_comment(raw.rstrip("\n")).rstrip()
            if not line.strip():
                continue
            if "\t" in line[:len(line) - len(line.lstrip())]:
                raise ValueError(f"{path}:{lineno}: tab indentation")
            indent = len(line) - len(line.lstrip(" "))
            key, sep, value = line.strip().partition(":")
            key = key.strip()
            if not sep or not key:
                raise ValueError(f"{path}:{lineno}: expected 'key: value', got {raw.strip()!r}")
            while stack and indent <= stack[-1][0]:
                close(stack.pop())
            want = (0 if not stack else stack[-1][2])
            if want is None:
                stack[-1][2] = want = indent
            if indent != want:
                raise ValueError(f"{path}:{lineno}: indentation {indent}, expected {want}")
            prefix = stack[-1][1] if stack else ""
            if prefix + key in flat:
                raise ValueError(f"{path}:{lineno}: {prefix + key} given twice")
            if value.strip():
                flat[prefix + key] = parse_scalar(value)
            else:
                stack.append([indent, prefix + key + ".", None])
    while stack:
        close(stack.pop())
    return flat


def _coerce(key: str, value, default):
    """`value` in the type of the default of `key`: 1e4 for an int setting is 10000; a value that does not fit
    (a fraction for an int, a word for a number or a flag) is an error."""
    if value is None or default is None:
        return value
    if isinstance(default, bool):
        if isinstance(value, bool):
            return value
    elif isinstance(default, int):
        if isinstance(value, int) and not isinstance(value, bool):
            return value
        if isinstance(value, float) and value.is_integer():
            return int(value)
    elif isinstance(default, float):
        if isinstance(value, (int, float)) and not isinstance(value, bool):
            return float(value)
    elif isinstance(default, str):
        if isinstance(value, (str, bool)):       # nerf.append_identity: a flag held as a truthy string
            return value
        if isinstance(value, (int, float)):
            return str(value)
    else:
        return value
    raise ValueError(f"{key}: {value!r} is not a {type(default).__name__}")


def merge(hparams: Dict[str, object], updates: Dict[str, object]) -> Dict[str, object]:
    """`updates` on top of `hparams`, each in the type of the value it replaces; unknown keys are an error (a typo
    would otherwise train with the default)."""
    unknown = sorted(set(updates) - set(hparams))
    if unknown:
        raise ValueError(f"unknown hyper-parameter(s): {', '.join(unknown)}")
    out = dict(hparams)
    out.update({k: _coerce(k, v, hparams[k]) for k, v in updates.items()})
    return out


def parse_overrides(opts: Sequence[str]) -> Dict[str, object]:
    """Trailing `key value` words of the command line."""
    if len(opts) % 2:
        raise ValueError(f"overrides come in 'key value' pairs, got {len(opts)} words")
    return {key: parse_scalar(value) for key, value in zip(opts[0::2], opts[1::2])}


def build_parser() -> argparse.ArgumentParser:
    p = argparse.ArgumentParser(prog="python -m mipnerf_pl_b200.fit", description=__doc__.split("\n\n")[0])
    p.add_argument("--data_path", type=str, required=True, help="data path.")
    p.add_argument("--out_dir", type=str, required=True, help="Output directory.")
    p.add_argument("--dataset_name", type=str, choices=list(DATASETS), required=True, help="Single or multi data.")
    p.add_argument("--config", type=str, default=None, help="Path to config file (default: the lego settings).")
    p.add_argument("--precision", type=str, choices=["bf16", "fp16"], default="bf16",
                   help="arithmetic of the training step's GEMMs")
    p.add_argument("opts", nargs=argparse.REMAINDER, help="Modify hparams, e.g. optimizer.max_steps 2000")
    return p


def parse_args(argv: Optional[Sequence[str]] = None):
    """(hparams, precision) from the command line; argparse errors exit with status 2."""
    parser = build_parser()
    args = parser.parse_args(argv)
    hp = default_hparams()
    try:
        if args.config:
            hp = merge(hp, read_config(args.config))
        hp = merge(hp, parse_overrides(args.opts))
    except (OSError, ValueError) as e:
        parser.error(str(e))
    hp.update(data_path=args.data_path, out_dir=args.out_dir, dataset_name=args.dataset_name)
    return hp, args.precision


# ---------------------------------------------------------------------------------------------------------------------
# checkpoints
# ---------------------------------------------------------------------------------------------------------------------
def checkpoint_dict(system: MipNeRFSystem, optimizer, scheduler, global_step: int, best: Dict[str, float]) -> dict:
    """The Lightning checkpoint layout (`state_dict` with the `mip_nerf.` prefix, `hyper_parameters`, `global_step`)
    plus what a resume needs: optimiser, scheduler, Philox state and the best-k bookkeeping."""
    model = system.mip_nerf
    return {
        "epoch": 0,
        "global_step": int(global_step),
        "state_dict": {k: v.detach().cpu() for k, v in system.state_dict().items()},
        "hyper_parameters": dict(system.hparams),
        "optimizer_states": [optimizer.state_dict()],
        "lr_schedulers": [scheduler.state_dict()],
        "rng_state": {"philox_seed": model.rng_seed, "philox_offset": model.rng_offset,
                      "torch": torch.get_rng_state(), "numpy": np.random.get_state(), "python": random.getstate()},
        "callbacks": {"ModelCheckpoint": {"monitor": "val/psnr", "mode": "max", "best_k_models": dict(best)}},
    }


def save_checkpoint(path: str, ckpt: dict) -> None:
    tmp = path + ".tmp"
    torch.save(ckpt, tmp)
    os.replace(tmp, path)


def _update_best(ckpt_dir: str, ckpt: dict, best: Dict[str, float], psnr: float, k: int = 2) -> None:
    """ModelCheckpoint(monitor='val/psnr', mode='max', save_top_k=2): keep the k best files, delete the one that drops."""
    if len(best) >= k and psnr <= min(best.values()):
        return
    path = os.path.join(ckpt_dir, f"epoch=0-step={ckpt['global_step']}.ckpt")
    best[path] = psnr
    while len(best) > k:
        worst = min(best, key=best.get)
        del best[worst]
        if os.path.exists(worst):
            os.remove(worst)
    ckpt["callbacks"]["ModelCheckpoint"]["best_k_models"] = dict(best)
    save_checkpoint(path, ckpt)


# ---------------------------------------------------------------------------------------------------------------------
# the driver
# ---------------------------------------------------------------------------------------------------------------------
def seed_everything(seed: int) -> None:
    torch.manual_seed(seed)
    torch.cuda.manual_seed_all(seed)
    np.random.seed(seed)
    random.seed(seed)


def _load_scene(hp: dict, split: str, white_bkgd: bool):
    from .datasets import load_blender_scene, load_multicam_scene
    if hp["dataset_name"] == "blender":
        return load_blender_scene(hp["data_path"], split, white_bkgd=white_bkgd)
    return load_multicam_scene(hp["data_path"], split, white_bkgd=white_bkgd)


def validate(system: MipNeRFSystem, hp: dict) -> float:
    """Mean fine PSNR of the first `val.sample_num` val images (limit_val_batches of the reference)."""
    from .datasets import dataset_dict
    from .metrics import evaluate
    ds = dataset_dict[hp["dataset_name"]](hp["data_path"], split="val", white_bkgd=hp["val.white_bkgd"],
                                          batch_type="single_image")
    psnrs, _ = evaluate(system, ds, max_images=int(hp["val.sample_num"]))
    return float(np.mean(psnrs))


def fit(hp: dict, precision: str = "bf16", stop_step: Optional[int] = None,
        log: Callable[[str], None] = print) -> dict:
    """Train `hp` to `optimizer.max_steps` (or `stop_step`, for a run cut short on purpose); returns
    {'global_step', 'val_psnr' (last validation), 'losses' [(step, loss, psnr)], 'ckpt_dir', 'system' (trained)}."""
    import torch.distributed as dist
    from .datasets import DeviceRayBank
    from .graph import GraphedTrainStep
    from .train import FusedAdam, MipLRDecay

    world = int(os.environ.get("WORLD_SIZE", "1"))
    if int(hp["num_gpus"]) > 1 and world != int(hp["num_gpus"]):
        raise RuntimeError(f"num_gpus={hp['num_gpus']}: launch with torchrun --nproc_per_node {hp['num_gpus']}")
    rank, local = int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1 and not dist.is_initialized():
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    seed_everything(int(hp["seed"]))

    system = MipNeRFSystem(hp, precision=precision).to(dev)
    model = system.mip_nerf
    optimizer = FusedAdam(model.parameters(), lr=hp["optimizer.lr_init"])
    scheduler = MipLRDecay(optimizer, hp["optimizer.lr_init"], hp["optimizer.lr_final"], hp["optimizer.max_steps"],
                           hp["optimizer.lr_delay_steps"], hp["optimizer.lr_delay_mult"])
    model.rng_seed, model.rng_offset = int(hp["seed"]) + rank, 0
    step, best = 0, {}
    ckpt_dir = os.path.join(hp["out_dir"], "ckpt", hp["exp_name"])
    resume = hp.get("checkpoint.resume_path")
    if resume:
        ck = torch.load(resume, map_location="cpu", weights_only=False)
        system.load_state_dict(ck["state_dict"])
        optimizer.load_state_dict(ck["optimizer_states"][0])
        scheduler.load_state_dict(ck["lr_schedulers"][0])
        step = int(ck["global_step"])
        model.rng_offset = int(ck["rng_state"]["philox_offset"])
        best = {path: v for path, v in ck["callbacks"]["ModelCheckpoint"]["best_k_models"].items()
                if os.path.dirname(os.path.abspath(path)) == os.path.abspath(ckpt_dir)}   # never delete another run's files
        log(f"resumed from {resume} at step {step}")
    if rank == 0:
        os.makedirs(ckpt_dir, exist_ok=True)

    bank = DeviceRayBank(_load_scene(hp, "train", hp["train.white_bkgd"]), dev)
    max_steps = int(hp["optimizer.max_steps"])
    stop = max_steps if stop_step is None else min(int(stop_step), max_steps)
    interval = max(1, int(hp["val.check_interval"]))
    trainer = GraphedTrainStep(model, optimizer, scheduler, bank, int(hp["train.batch_size"]),
                               randomized=bool(hp["train.randomized"]), white_bkgd=bool(hp["train.white_bkgd"]),
                               coarse_loss_mult=float(hp["loss.coarse_loss_mult"]),
                               disable_multiscale_loss=bool(hp["loss.disable_multiscale_loss"]),
                               num_steps=max_steps, ring_len=interval, world=world)
    losses, val_psnr = [], None
    while step < stop:
        k = min(interval - step % interval, stop - step)
        trainer.replay(k)
        rows = trainer.sync()
        step += k
        losses.extend(rows)
        if rows:
            log(f"step {step}: train/loss {rows[-1][1]:.6f} train/psnr {rows[-1][2]:.3f}")
        if step % interval == 0 or step == max_steps:
            if rank == 0:
                system.eval()
                val_psnr = validate(system, hp)
                ckpt = checkpoint_dict(system, optimizer, scheduler, step, best)
                _update_best(ckpt_dir, ckpt, best, val_psnr)
                save_checkpoint(os.path.join(ckpt_dir, "last.ckpt"), ckpt)
                log(f"step {step}: val/psnr {val_psnr:.3f}")
            if world > 1:
                dist.barrier()
    return {"global_step": step, "val_psnr": val_psnr, "losses": losses, "ckpt_dir": ckpt_dir, "system": system}


def main(argv: Optional[Sequence[str]] = None) -> int:
    hp, precision = parse_args(argv)
    fit(hp, precision=precision)
    return 0


if __name__ == "__main__":
    sys.exit(main())
