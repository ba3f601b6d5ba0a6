"""Eager vs graph-captured training step (`GraphedTrainStep`) on one GPU: ms per step with CUDA events over
--steps steps of each, alternating eager / graphed blocks, at each --rays batch, on a device-resident synthetic scene.
The eager step is what a hand-written loop does: `DeviceRayBank.sample`, `forward_backward` (in-kernel Philox),
`FusedAdam.step`, `MipLRDecay.step`; it never reads the loss back (no host sync).  Prints and writes one JSON
document with the card name and power limit read in the same run.

    python tools/train_graph_bench.py [--rays 4096 1024] [--steps 200] [--precision bf16] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import mipnerf_pl_b200 as mp  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def trainee(precision, dev):
    model = mp.MipNerf(precision=precision)
    model.load_state_dict(mp.make_state_dict(seed=0, kind="xavier"))
    model = model.to(dev)
    model.rng_seed, model.rng_offset = 4, 0
    opt = mp.FusedAdam(model.parameters(), lr=5e-4)
    sched = mp.MipLRDecay(opt, 5e-4, 5e-6, 1000000, 2500, 0.01)
    return model, opt, sched


def timed(fn, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn(steps)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rays", type=int, nargs="+", default=[4096, 1024])
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--repeats", type=int, default=3, help="alternating eager / graphed blocks of --steps steps")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp16"])
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("train_graph_bench: needs a GPU")
    dev = torch.device("cuda", 0)
    with tempfile.TemporaryDirectory() as root:
        mp.write_synthetic_blender_scene(root, n_images=8, height=200, width=200, seed=0, splits=("train",))
        bank = mp.DeviceRayBank(mp.load_blender_scene(root, "train", white_bkgd=True), dev)
    rows = []
    for b in args.rays:
        em, eo, es = trainee(args.precision, dev)
        gm, go, gs = trainee(args.precision, dev)
        total = (args.repeats + 1) * args.steps + 8
        graphed = mp.GraphedTrainStep(gm, go, gs, bank, b, num_steps=total, ring_len=args.steps)

        def eager(k):
            for _ in range(k):
                rays, rgb = bank.sample(b)
                mp.forward_backward(em, rays, rgb, True, True)
                eo.step()
                es.step()

        def replay(k):
            graphed.replay(k)

        eager(3)
        replay(3)
        torch.cuda.synchronize()
        e_ms, g_ms = [], []
        for _ in range(args.repeats):
            e_ms.append(timed(eager, args.steps))
            g_ms.append(timed(replay, args.steps))
        logged = graphed.sync()
        row = {"rays_per_gpu": b, "steps_per_block": args.steps, "blocks": args.repeats,
               "eager_ms_per_step": e_ms, "graphed_ms_per_step": g_ms,
               "eager_ms_median": float(np.median(e_ms)), "graphed_ms_median": float(np.median(g_ms)),
               "saving_ms_per_step": float(np.median(e_ms) - np.median(g_ms)),
               "last_logged": {"step": logged[-1][0], "loss": logged[-1][1], "psnr": logged[-1][2]}}
        print(json.dumps(row), flush=True)
        rows.append(row)
        del graphed
        torch.cuda.empty_cache()
    doc = {"what": "training step, eager (host-driven) vs one CUDA graph per step (GraphedTrainStep)",
           "precision": args.precision, "gpu": card(), "torch": torch.__version__, "cuda": torch.version.cuda,
           "timing": "CUDA events around --steps back-to-back steps, blocks alternating eager / graphed",
           "results": rows}
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
