"""The training driver's host side without a GPU: the config reader and CLI of `python -m mipnerf_pl_b200.fit`, the
per-step Adam tables of the captured training step, the checkpoint writer, and the promise that the device-driven
training step left the inference level kernels' code untouched."""
import contextlib
import ctypes as C
import ctypes.util
import json
import os
import warnings

import numpy as np
import pytest
import torch

from helpers import GOLDEN

import mipnerf_pl_b200 as mp
from mipnerf_pl_b200 import fit as F
from mipnerf_pl_b200.train import adam_tables

LEGO = """seed: 4
num_gpus: 1
exp_name: 'lego'
train:
  batch_size: 3072
  batch_type: 'all_images'  # rays sampled from every image
  num_work: 4
  randomized: True
  white_bkgd: True
val:
  batch_size: 1
  batch_type: 'single_image'
  num_work: 4
  randomized: False
  white_bkgd: True
  check_interval: 10000
  chunk_size: 8192  # rays per forward
  sample_num: 4
nerf:
  num_samples: 128
  num_levels: 2
  resample_padding: 0.01
  stop_resample_grad: True
  use_viewdirs: True
  disparity: False
  ray_shape: 'cone'
  min_deg_point: 0
  max_deg_point: 16
  deg_view: 4
  density_activation: 'softplus'
  density_noise: 0.
  density_bias: -1.
  rgb_activation: 'sigmoid'
  rgb_padding: 0.001
  disable_integration: False
  append_identity: Ture
  mlp:
    net_depth: 8
    net_width: 256
    net_depth_condition: 1
    net_width_condition: 128
    net_activation: 'relu'
    skip_index: 4
    num_rgb_channels: 3
    num_density_channels: 1
optimizer:
  lr_init: 5e-4
  lr_final: 5e-6
  lr_delay_steps: 2500
  lr_delay_mult: 0.01
  max_steps: 1000000
loss:
  disable_multiscale_loss: False
  coarse_loss_mult: 0.1
checkpoint:
  resume_path: None
"""


@pytest.fixture
def lego(tmp_path):
    path = tmp_path / "lego.yaml"
    path.write_text(LEGO)
    return str(path)


def test_config_file_reads_as_default_hparams(lego):
    cfg = F.read_config(lego)
    want = mp.default_hparams()
    assert cfg == want
    assert [type(cfg[k]) for k in want] == [type(v) for v in want.values()]


def test_cli_config_and_overrides(lego, tmp_path):
    hp, precision = F.parse_args(["--data_path", str(tmp_path), "--out_dir", "out", "--dataset_name", "multi_blender",
                                  "--config", lego, "optimizer.max_steps", "2000", "train.randomized", "False",
                                  "exp_name", "'chair'", "nerf.density_noise", "1e-1", "checkpoint.resume_path",
                                  "out/last.ckpt"])
    assert precision == "bf16"
    assert hp["optimizer.max_steps"] == 2000 and hp["train.randomized"] is False and hp["exp_name"] == "chair"
    assert hp["nerf.density_noise"] == 0.1 and hp["checkpoint.resume_path"] == "out/last.ckpt"
    assert hp["data_path"] == str(tmp_path) and hp["out_dir"] == "out" and hp["dataset_name"] == "multi_blender"
    changed = {"optimizer.max_steps", "train.randomized", "exp_name", "nerf.density_noise", "checkpoint.resume_path",
               "data_path", "out_dir", "dataset_name"}
    base = mp.default_hparams()
    assert {k: v for k, v in hp.items() if k not in changed} == {k: v for k, v in base.items() if k not in changed}


@pytest.mark.parametrize("argv", [
    [],                                                                                  # required arguments missing
    ["--data_path", "d", "--out_dir", "o"],
    ["--data_path", "d", "--out_dir", "o", "--dataset_name", "llff"],                    # not a dataset of the project
    ["--data_path", "d", "--out_dir", "o", "--dataset_name", "blender", "train.batch_size"],   # odd override list
    ["--data_path", "d", "--out_dir", "o", "--dataset_name", "blender", "train.batchsize", "8"],  # unknown key
    ["--data_path", "d", "--out_dir", "o", "--dataset_name", "blender", "--precision", "fp32"],   # no graphed fp32 step
    ["--data_path", "d", "--out_dir", "o", "--dataset_name", "blender", "--config", "/nonexistent.yaml"],
])
def test_cli_rejects_bad_arguments(argv, capsys):
    with pytest.raises(SystemExit) as e:
        F.parse_args(argv)
    assert e.value.code == 2
    assert "error" in capsys.readouterr().err


def test_config_reader_rejects_malformed_files(tmp_path):
    for text in ("train:\n  batch_size 3072\n", "train:\n\tbatch_size: 1\n", "seed: 4\nnot a mapping\n"):
        p = tmp_path / "bad.yaml"
        p.write_text(text)
        with pytest.raises(ValueError):
            F.read_config(str(p))
    p = tmp_path / "extra.yaml"
    p.write_text("train:\n  batchsize: 8\n")
    with pytest.raises(ValueError, match="train.batchsize"):
        F.merge(mp.default_hparams(), F.read_config(str(p)))


@pytest.mark.parametrize("hp", [dict(), dict(lr_init=1e-3, lr_final=1e-5, max_steps=40, lr_delay_steps=0,
                                              lr_delay_mult=1.0)])
def test_adam_tables_equal_fused_adam_host_math(hp):
    """Entry t of the tables is what FusedAdam's update t hands the library when MipLRDecay drives its lr:
    (float)(lr / (1 - b1^t)) and (float)sqrt(1 - b2^t), evaluated in double with the C library's pow."""
    kw = dict(lr_init=5e-4, lr_final=5e-6, max_steps=1000000, lr_delay_steps=2500, lr_delay_mult=0.01)
    kw.update(hp)
    n = 60
    libm = C.CDLL(ctypes.util.find_library("m"))
    libm.pow.restype, libm.pow.argtypes = C.c_double, [C.c_double, C.c_double]
    opt = mp.FusedAdam([torch.nn.Parameter(torch.zeros(2))], lr=kw["lr_init"], betas=(0.9, 0.999))
    with _quiet():
        sched = mp.MipLRDecay(opt, kw["lr_init"], kw["lr_final"], kw["max_steps"], kw["lr_delay_steps"],
                              kw["lr_delay_mult"])
    step_size, bc2_sqrt = adam_tables(n, (0.9, 0.999), **kw)
    assert step_size.dtype == np.float32 and step_size.shape == (n + 1,)
    for t in range(1, n + 1):
        lr = opt.param_groups[0]["lr"]
        want_ss = C.c_float(lr / (1.0 - libm.pow(0.9, float(t)))).value
        want_b2 = C.c_float((1.0 - libm.pow(0.999, float(t))) ** 0.5).value
        assert step_size[t].tobytes() == np.float32(want_ss).tobytes(), t
        assert bc2_sqrt[t].tobytes() == np.float32(want_b2).tobytes(), t
        with _quiet():   # the optimiser never steps here: torch warns about the order
            sched.step()


@contextlib.contextmanager
def _quiet():
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        yield


def test_checkpoint_writer_output_loads(tmp_path):
    hp = mp.default_hparams(data_path=str(tmp_path), out_dir=str(tmp_path), dataset_name="blender")
    system = mp.MipNeRFSystem(hp)
    torch.manual_seed(3)
    for p in system.parameters():
        p.data.normal_()
    model = system.mip_nerf
    model.rng_seed, model.rng_offset = 4, 17
    opt = mp.FusedAdam(model.parameters(), lr=5e-4)
    for p in model.parameters():
        opt.state[p] = {"step": 17, "exp_avg": torch.rand_like(p), "exp_avg_sq": torch.rand_like(p)}
    with _quiet():
        sched = mp.MipLRDecay(opt, 5e-4, 5e-6, 1000, 10, 0.01)
    best = {}
    ckpt_dir = str(tmp_path / "ckpt" / "lego")
    os.makedirs(ckpt_dir)
    for step, psnr in ((100, 20.0), (200, 22.0), (300, 21.0), (400, 19.0)):
        ck = F.checkpoint_dict(system, opt, sched, step, best)
        F._update_best(ckpt_dir, ck, best, psnr)
        F.save_checkpoint(os.path.join(ckpt_dir, "last.ckpt"), ck)
    assert sorted(os.listdir(ckpt_dir)) == ["epoch=0-step=200.ckpt", "epoch=0-step=300.ckpt", "last.ckpt"]
    loaded = mp.MipNeRFSystem.load_from_checkpoint(os.path.join(ckpt_dir, "last.ckpt"))
    for (k, v), (k2, v2) in zip(system.state_dict().items(), loaded.state_dict().items()):
        assert k == k2 and k.startswith("mip_nerf.") and torch.equal(v, v2)
    raw = torch.load(os.path.join(ckpt_dir, "last.ckpt"), weights_only=False)
    assert raw["global_step"] == 400 and raw["hyper_parameters"] == hp
    assert raw["rng_state"]["philox_offset"] == 17
    assert raw["optimizer_states"][0]["state"][0]["step"] == 17
    assert set(raw["callbacks"]["ModelCheckpoint"]["best_k_models"].values()) == {22.0, 21.0}
    opt2 = mp.FusedAdam(loaded.mip_nerf.parameters(), lr=1.0)
    opt2.load_state_dict(raw["optimizer_states"][0])
    p0 = next(loaded.mip_nerf.parameters())
    assert torch.equal(opt2.state[p0]["exp_avg"], opt.state[next(model.parameters())]["exp_avg"])


def test_pixel_id_mirror_is_philox_and_in_range():
    """The host mirror of the device batch sampler: Philox4x32-10's published known-answer vectors, ids in range."""
    from mipnerf_pl_b200.datasets import philox4x32_10_first
    assert int(philox4x32_10_first(0, 0, 0, 0, 0, 0)) == 0x6627E8D5
    assert int(philox4x32_10_first(*([0xFFFFFFFF] * 6))) == 0x408F276D
    assert int(philox4x32_10_first(0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344, 0xA4093822, 0x299F31D0)) == 0xD16CFE09
    ids = mp.philox_pixel_ids(4, 7, 100000, 1000)
    assert ids.min() >= 0 and ids.max() < 1000 and len(np.unique(ids)) == 1000
    assert not np.array_equal(ids, mp.philox_pixel_ids(4, 8, 100000, 1000))
    assert np.array_equal(ids[50:], mp.philox_pixel_ids(4, 7, 100000 - 50, 1000, ray_base=50))
    assert mp.philox_pixel_ids(1, 2, 4, 1 << 32).max() < 1 << 32


def test_inference_level_kernels_keep_their_code():
    """The device-state reads of the training step live in the kTrain instantiation only: every other instantiation
    of the level kernels keeps the opcode stream and register count of the library before that change
    (tests/golden/level_kernel_sass.json, recorded with tools/sass_opcodes.py)."""
    import __graft_entry__ as ge
    from tools import sass_opcodes
    try:
        sass_opcodes.cuobjdump()
    except FileNotFoundError:
        pytest.skip("no cuobjdump")
    ge.build()
    want = json.load(open(os.path.join(GOLDEN, "level_kernel_sass.json")))
    got = sass_opcodes.digest()
    inference = [k for k in want if "ELb1ELb0ELb0EE" not in k]   # <kFmt, kPair, kX3, kTrain=1, kTS=0, kNoise=0>
    assert len(inference) == 16 and "mlp_level_kernelILi1ELb1ELb0ELb0ELb0ELb0EEEvNS0_11LevelParamsE" in inference
    for k in inference:
        assert got.get(k) == want[k], k


@pytest.mark.parametrize("precision", ["fp32", "fp16x3", "bf16x3"])
def test_graphed_step_is_bf16_fp16_only(precision):
    model = mp.MipNerf(precision=precision)
    opt = mp.FusedAdam(model.parameters(), lr=5e-4)
    with _quiet():
        sched = mp.MipLRDecay(opt, 5e-4, 5e-6, 100, 0, 1.0)
    with pytest.raises(NotImplementedError):
        mp.GraphedTrainStep(model, opt, sched, None, 64)


def test_config_reader_indentation_and_empty_values(tmp_path):
    p = tmp_path / "c.yaml"
    p.write_text("a:\n    b: 1\n  c: 2\n")                       # a dedent that matches no open section
    with pytest.raises(ValueError, match="indentation"):
        F.read_config(str(p))
    p.write_text("a:\n  b: 1\n  b: 2\n")
    with pytest.raises(ValueError, match="twice"):
        F.read_config(str(p))
    p.write_text("checkpoint:\n  resume_path:\nloss:\n  coarse_loss_mult: 0.1\n")
    assert F.read_config(str(p)) == {"checkpoint.resume_path": None, "loss.coarse_loss_mult": 0.1}
    p.write_text("checkpoint:\n  resume_path:  # none yet\n")
    assert F.read_config(str(p)) == {"checkpoint.resume_path": None}


def test_overrides_take_the_type_of_the_default(lego, tmp_path):
    hp, _ = F.parse_args(["--data_path", "d", "--out_dir", "o", "--dataset_name", "blender", "--config", lego,
                          "optimizer.max_steps", "1e4", "val.check_interval", "2500.0", "nerf.density_noise", "1",
                          "exp_name", "7", "nerf.append_identity", "True"])
    assert hp["optimizer.max_steps"] == 10000 and type(hp["optimizer.max_steps"]) is int
    assert type(hp["val.check_interval"]) is int and hp["nerf.density_noise"] == 1.0
    assert type(hp["nerf.density_noise"]) is float and hp["exp_name"] == "7" and hp["nerf.append_identity"] is True
    for bad in (["optimizer.max_steps", "1.5"], ["train.randomized", "1"], ["nerf.density_noise", "abc"]):
        with pytest.raises(ValueError, match=bad[0]):
            F.merge(mp.default_hparams(), F.parse_overrides(bad))
