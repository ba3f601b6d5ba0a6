"""The captured training step (`GraphedTrainStep`) and the driver on top of it (`fit`), on the GPU.

The graphed step must be the eager step, bit for bit: eager = `DeviceRayBank.rays` on the pixel ids recomputed on the
host from Philox, `forward_backward` with (seed, offset + i), `FusedAdam` + `MipLRDecay`."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp_

import mipnerf_pl_b200 as mp
from mipnerf_pl_b200 import fit as F

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def scene_dir(tmp_path_factory):
    root = str(tmp_path_factory.mktemp("scene"))
    mp.write_synthetic_blender_scene(root, n_images=4, height=40, width=32, seed=1)
    return root


@pytest.fixture(scope="module")
def bank(scene_dir):
    return mp.DeviceRayBank(mp.load_blender_scene(scene_dir, "train", white_bkgd=True), DEV)


def _trainee(precision, density_noise, seed=11, dev=DEV):
    model = mp.MipNerf(precision=precision, density_noise=density_noise)
    model.load_state_dict(mp.make_state_dict(seed=3, kind="xavier"))
    model = model.to(dev)
    model.rng_seed, model.rng_offset = seed, 0
    opt = mp.FusedAdam(model.parameters(), lr=5e-4)
    sched = mp.MipLRDecay(opt, 5e-4, 5e-6, 1000, 3, 0.01)
    return model, opt, sched


def _eager_step(model, opt, sched, bank, b, allreduce=False):
    ids = mp.philox_pixel_ids(model.rng_seed, model.rng_offset, b, bank.num_pixels)
    rays, rgb = bank.rays(torch.from_numpy(ids))
    out = mp.forward_backward(model, rays, rgb, True, True)       # draws (seed, offset), then offset += 1
    if allreduce:
        mp.allreduce_grads(model.parameters())                    # DDP: the mean of the ranks' gradients
    opt.step()
    sched.step()
    return ids, float(out["loss"]), float(mp.calc_psnr(out["ret"][-1][0], rgb))


def _assert_same_state(a, oa, b, ob):
    for (n, pa), pb in zip(a.named_parameters(), b.parameters()):
        assert torch.equal(pa, pb), n
        assert torch.equal(oa.state[pa]["exp_avg"], ob.state[pb]["exp_avg"]), n
        assert torch.equal(oa.state[pa]["exp_avg_sq"], ob.state[pb]["exp_avg_sq"]), n
        assert oa.state[pa]["step"] == ob.state[pb]["step"], n


@pytest.mark.parametrize("precision", ["bf16", "fp16"])
@pytest.mark.parametrize("density_noise", [0.0, 0.5])
def test_graphed_steps_equal_eager_steps(bank, precision, density_noise):
    b, k = 512, 5
    ga, oa, sa = _trainee(precision, density_noise)
    eb, ob, sb = _trainee(precision, density_noise)
    step = mp.GraphedTrainStep(ga, oa, sa, bank, b, num_steps=50, ring_len=8)
    step.replay(k)
    rows = step.sync()
    eager = [_eager_step(eb, ob, sb, bank, b) for _ in range(k)]
    assert [r[0] for r in rows] == list(range(1, k + 1))
    assert [r[1] for r in rows] == [e[1] for e in eager], "per-step losses"
    np.testing.assert_allclose([r[2] for r in rows], [e[2] for e in eager], rtol=1e-6)
    assert np.array_equal(step.batch[2].cpu().numpy(), eager[-1][0]), "pixel ids of the last step"
    _assert_same_state(ga, oa, eb, ob)
    assert ga.rng_offset == eb.rng_offset == k and sa.last_epoch == sb.last_epoch == k
    assert oa.param_groups[0]["lr"] == ob.param_groups[0]["lr"]
    # K graphed steps + sync + one eager step == K + 1 eager steps
    _eager_step(ga, oa, sa, bank, b)
    _eager_step(eb, ob, sb, bank, b)
    _assert_same_state(ga, oa, eb, ob)
    losses = [r[1] for r in rows]
    assert all(np.isfinite(losses))


def test_pixel_sampler_is_philox_uniform_generator(bank):
    """The ids come from the generator of mipnerf_b200_philox_uniform (stream 64): its 24-bit uniforms are the top
    bits of the host mirror's 32-bit words, and the device ids equal the mirror's."""
    from mipnerf_pl_b200.datasets import philox4x32_10_first
    seed, offset, n = 0x1234_5678_9ABC, 9, 4096
    u = mp.philox_uniform(seed, offset, 64, n, 1, DEV).reshape(-1).cpu().numpy()
    g = np.arange(n, dtype=np.uint64)
    x = philox4x32_10_first(g & 0xFFFFFFFF, g >> np.uint64(32), 64 << 24, offset, seed & 0xFFFFFFFF,
                            (seed >> 32) ^ (offset >> 32))
    scale = np.float32(1.0) - np.float32(2.0 ** -23)                 # stream != 0: uniform_(to = 1/ncols - eps)
    assert np.array_equal(u, ((x >> 8).astype(np.float32) * np.float32(2.0 ** -24)) * scale)
    state = torch.tensor([seed, offset], dtype=torch.int64, device=DEV)
    rays, rgb, ids = bank.sample_philox(state, n, ray_base=100)
    want = mp.philox_pixel_ids(seed, offset, n, bank.num_pixels, ray_base=100)
    assert np.array_equal(ids.cpu().numpy(), want)
    r2, rgb2 = bank.rays(torch.from_numpy(want))
    assert all(torch.equal(a, c) for a, c in zip(rays, r2)) and torch.equal(rgb, rgb2)


def _hp(scene_dir, out_dir, **over):
    hp = mp.default_hparams(data_path=scene_dir, out_dir=out_dir, dataset_name="blender")
    hp.update({"train.batch_size": 1024, "val.check_interval": 100, "val.sample_num": 1, "val.chunk_size": 4096,
               "optimizer.max_steps": 200, "optimizer.lr_delay_steps": 20})
    hp.update(over)
    return hp


def test_fit_trains_checkpoints_and_resumes(scene_dir, tmp_path):
    logs = []
    full = F.fit(_hp(scene_dir, str(tmp_path / "a")), log=logs.append)
    assert full["global_step"] == 200 and len(full["losses"]) == 200
    losses = np.array([r[1] for r in full["losses"]])
    # the synthetic scene is random RGBA noise: the loss falls by ~11 % over 200 steps (0.186 -> 0.165) and floors at
    # the colours' variance
    assert np.isfinite(losses).all() and losses[-20:].mean() < 0.95 * losses[:20].mean(), (losses[:20], losses[-20:])
    ckpt_dir = full["ckpt_dir"]
    assert sorted(os.listdir(ckpt_dir)) == ["epoch=0-step=100.ckpt", "epoch=0-step=200.ckpt", "last.ckpt"]
    system = mp.MipNeRFSystem.load_from_checkpoint(os.path.join(ckpt_dir, "last.ckpt"), precision="bf16").to(DEV)
    val = mp.Blender(scene_dir, split="val", white_bkgd=True, batch_type="single_image")
    psnrs, ssims = mp.evaluate(system, val, max_images=1)
    assert np.isfinite(psnrs).all() and abs(psnrs[0] - full["val_psnr"]) < 1e-3
    # resume from the step-100 checkpoint: steps 101..200 again, same parameters as the uninterrupted run
    resumed = F.fit(_hp(scene_dir, str(tmp_path / "b"),
                        **{"checkpoint.resume_path": os.path.join(ckpt_dir, "epoch=0-step=100.ckpt")}), log=logs.append)
    assert resumed["global_step"] == 200 and [r[0] for r in resumed["losses"]] == list(range(101, 201))
    assert [r[1] for r in resumed["losses"]] == [r[1] for r in full["losses"][100:]]
    a = torch.load(os.path.join(ckpt_dir, "last.ckpt"), weights_only=False)
    b = torch.load(os.path.join(resumed["ckpt_dir"], "last.ckpt"), weights_only=False)
    for k, v in a["state_dict"].items():
        assert torch.equal(v, b["state_dict"][k]), k
    assert os.path.exists(os.path.join(ckpt_dir, "epoch=0-step=100.ckpt")), "a resumed run leaves other runs' files"


def _two_rank_worker(rank, world, port, scene, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), LOCAL_RANK=str(rank),
                      WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        res = {}
        bank = mp.DeviceRayBank(mp.load_blender_scene(scene, "train", white_bkgd=True), dev)
        b, k = 512, 4
        ga, oa, sa = _trainee("bf16", 0.5, seed=11 + rank, dev=dev)       # every rank its own batch and draws
        eb, ob, sb = _trainee("bf16", 0.5, seed=11 + rank, dev=dev)
        step = mp.GraphedTrainStep(ga, oa, sa, bank, b, num_steps=50, ring_len=8, world=world)
        step.replay(k)
        rows = step.sync()
        eager = [_eager_step(eb, ob, sb, bank, b, allreduce=True) for _ in range(k)]
        res["losses"] = [r[1] for r in rows] == [e[1] for e in eager]
        try:
            _assert_same_state(ga, oa, eb, ob)
            res["state"] = True
        except AssertionError as e:
            res["state"] = str(e)
        res["steps"] = oa.state[next(ga.parameters())]["step"] == k and ga.rng_offset == k

        def replicas_agree(model):
            flat = torch.cat([p.detach().reshape(-1) for p in model.parameters()])
            got = [torch.empty_like(flat) for _ in range(world)]
            dist.all_gather(got, flat)
            return all(torch.equal(got[0], g) for g in got[1:])

        res["replicas"] = replicas_agree(ga)
        # the driver under torchrun-style ranks: 40 steps, validation and checkpoints on rank 0
        hp = _hp(scene, os.path.join(out_dir, "fit"), num_gpus=world, **{
            "train.batch_size": 512, "val.check_interval": 20, "optimizer.max_steps": 40})
        out = F.fit(hp, log=lambda *_: None)
        res["fit"] = (out["global_step"] == 40 and len(out["losses"]) == 40 and
                      bool(np.isfinite([r[1] for r in out["losses"]]).all()))
        res["fit_replicas"] = replicas_agree(out["system"].mip_nerf)
        if rank == 0:
            res["fit_ckpt"] = os.path.exists(os.path.join(out["ckpt_dir"], "last.ckpt"))
        torch.save(res, os.path.join(out_dir, f"res{rank}.pt"))
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs (NCCL)")
def test_graphed_step_with_allreduce_equals_eager_ddp_on_two_gpus(scene_dir, tmp_path):
    """GraphedTrainStep(world=2): the NCCL all-reduce captured in the graph, per-rank batches (seed + rank), equals
    eager forward_backward + allreduce_grads + FusedAdam + MipLRDecay on every rank bit for bit; the replicas stay
    identical; fit() runs with num_gpus=2."""
    world = 2
    port = 31500 + (os.getpid() % 2000)
    mp_.spawn(_two_rank_worker, args=(world, port, scene_dir, str(tmp_path)), nprocs=world, join=True)
    for r in range(world):
        res = torch.load(tmp_path / f"res{r}.pt")
        print(f"rank {r}: {res}")
        assert res["losses"] and res["state"] is True and res["steps"], res
        assert res["replicas"] and res["fit"] and res["fit_replicas"], res
    assert torch.load(tmp_path / "res0.pt")["fit_ckpt"]
