"""CPU-side tests: the C-ABI library loads and exports every declared symbol, the host mirror keeps
the reference's API/state_dict layout, helpers behave, and errors surface without a GPU."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from helpers import ROOT, make_state_dict, oracle

import mipnerf_pl_b200 as mp
from mipnerf_pl_b200 import _cabi


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    return _cabi.lib()


def test_header_symbols_all_exported(lib):
    header = open(os.path.join(ROOT, "include", "mipnerf_b200.h")).read()
    declared = set(re.findall(r"\b(mipnerf_b200_[a-z0-9_]+)\s*\(", header))
    assert declared, "no prototypes parsed"
    assert declared == set(_cabi.EXPORTED_SYMBOLS), declared ^ set(_cabi.EXPORTED_SYMBOLS)
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.mipnerf_b200_abi_version() == _cabi.ABI_VERSION == 4


def test_ctypes_structs_match_header_layout():
    assert C.sizeof(_cabi.Linear) == 24
    assert C.sizeof(_cabi.Config) == 19 * 4
    assert C.sizeof(_cabi.RaysStruct) == 7 * 8
    assert C.sizeof(_cabi.LevelOut) == 7 * 8
    assert C.sizeof(_cabi.Weights) == 8 + 4 + 4 + 8 + 8
    assert C.sizeof(_cabi.LinearGrad) == 16
    assert C.sizeof(_cabi.Loss) == 8 * 8


def test_argument_validation_without_gpu(lib):
    cfg = mp.MipNerf()._config()
    assert lib.mipnerf_b200_workspace_bytes(C.byref(cfg), 4096, _cabi.FP32) > 1 << 30
    assert lib.mipnerf_b200_workspace_bytes(C.byref(cfg), 10 ** 9, _cabi.FP32) == \
        lib.mipnerf_b200_workspace_bytes(C.byref(cfg), 4096, _cabi.FP32), "scratch is bounded by the chunk size"
    bad = mp.MipNerf(num_samples=100)._config()
    assert lib.mipnerf_b200_workspace_bytes(C.byref(bad), 16, _cabi.FP32) == 0
    rc = lib.mipnerf_b200_forward(C.byref(bad), None, None, 0, None, None, 1, 0, None, None, 0, None)
    assert rc == _cabi.EUNSUPPORTED and b"num_samples" in lib.mipnerf_b200_last_error()
    rc = lib.mipnerf_b200_forward(C.byref(cfg), None, None, 0, None, None, 1, 0, None, None, 0, None)
    assert rc == _cabi.EINVAL
    # density_noise (models/mip_nerf.py:232-233) travels in the config: a negative / non-finite std is a bad argument
    assert abs(mp.MipNerf(density_noise=0.25)._config().density_noise - 0.25) < 1e-7
    for std in (-1.0, float("nan"), float("inf")):
        neg = mp.MipNerf(density_noise=std)._config()
        assert lib.mipnerf_b200_workspace_bytes(C.byref(neg), 16, _cabi.FP32) == 0
        rc = lib.mipnerf_b200_forward(C.byref(neg), None, None, 0, None, None, 1, 0, None, None, 0, None)
        assert rc == _cabi.EINVAL and b"density_noise" in lib.mipnerf_b200_last_error(), std
    rc = lib.mipnerf_b200_philox_normal(None, 0, 4, 128, None, None)
    assert rc == _cabi.EINVAL
    # tensor-core shape contract (include/mipnerf_b200.h): the operand image exists for the shipped architecture with
    # max_deg_point 1..16 / deg_view 1..4 (narrower encodings add the zero-padded fp32 copies: 603 KB), not otherwise
    base = lib.mipnerf_b200_packed_weights_bytes(C.byref(cfg), _cabi.BF16)
    assert base > 0 and lib.mipnerf_b200_packed_weights_bytes(C.byref(cfg), _cabi.FP32) == 0
    for kw in (dict(max_deg_point=10), dict(deg_view=2), dict(max_deg_point=1, deg_view=1)):
        narrow = mp.MipNerf(**kw)._config()
        nb = lib.mipnerf_b200_packed_weights_bytes(C.byref(narrow), _cabi.BF16)
        assert base < nb <= base + 604 * 1024 + 256, (kw, nb - base)
        assert lib.mipnerf_b200_workspace_bytes(C.byref(narrow), 4096, _cabi.BF16) == \
            lib.mipnerf_b200_workspace_bytes(C.byref(cfg), 4096, _cabi.BF16)
    for kw in (dict(min_deg_point=1), dict(max_deg_point=17), dict(num_samples=64), dict(mlp_net_width=128),
               dict(mlp_net_depth=6), dict(use_viewdirs=False, mlp_net_width_condition=256)):
        other = mp.MipNerf(**kw)._config()
        assert lib.mipnerf_b200_packed_weights_bytes(C.byref(other), _cabi.BF16) == 0, kw
        assert lib.mipnerf_b200_workspace_bytes(C.byref(other), 16, _cabi.FP32) > 0, kw      # the fp32 path takes it
    with pytest.raises(NotImplementedError):
        _cabi.check(_cabi.EUNSUPPORTED, "x")
    with pytest.raises(ValueError):
        _cabi.check(_cabi.EINVAL, "x")


def test_cpu_tensors_are_rejected_no_fallback():
    model = mp.MipNerf()
    rays = mp.random_ray_batch(8, seed=0)
    with pytest.raises(RuntimeError, match="CUDA"):
        model(rays, False, True)
    with pytest.raises(RuntimeError, match="CUDA"):
        mp.pos_enc(rays.viewdirs, 0, 4)


def test_state_dict_layout_matches_reference_keys():
    model = mp.MipNerf()
    keys = list(model.state_dict().keys())
    want = list(make_state_dict(0).keys())
    assert keys == want
    assert sum(p.numel() for p in model.parameters()) == 612740        # SURVEY.md §8a
    shapes = {k: tuple(v.shape) for k, v in model.state_dict().items()}
    assert shapes["mlp.layers.5.0.weight"] == (256, 352) and shapes["mlp.view_layers.0.0.weight"] == (128, 283)
    system = mp.MipNeRFSystem(mp.default_hparams())
    assert all(k.startswith("mip_nerf.mlp.") for k in system.state_dict())
    assert len(system.state_dict()) == 24


def test_checkpoint_roundtrip(tmp_path):
    system = mp.MipNeRFSystem(mp.default_hparams())
    sd = {"mip_nerf." + k: v for k, v in make_state_dict(3).items()}
    ckpt = {"state_dict": sd, "hyper_parameters": mp.default_hparams(), "epoch": 27, "global_step": 329999}
    path = tmp_path / "epoch=27-step=329999.ckpt"
    torch.save(ckpt, path)
    loaded = mp.MipNeRFSystem.load_from_checkpoint(str(path))
    for k, v in loaded.state_dict().items():
        assert torch.equal(v, sd[k])
    assert loaded.val_chunk_size == 8192


def test_unsupported_modes_raise_like_reference():
    with pytest.raises(NotImplementedError):
        mp.MipNerf(rgb_activation="tanh")
    with pytest.raises(NotImplementedError):
        mp.MipNerf(density_activation="relu")
    with pytest.raises(NotImplementedError):
        mp.MipNerf(mlp_net_activation="gelu")


def test_rearrange_render_image_chunks():
    h, w = 5, 7
    full = mp.blender_rays(mp.spheric_pose(0.3), height=800, width=800)
    sub = mp.Rays(*[f[:h, :w][None] for f in full])
    rays = mp.rays_to_torch(sub, flatten=False)
    chunks, mask = mp.rearrange_render_image(rays, 8)
    assert [c.origins.shape[0] for c in chunks] == [8, 8, 8, 8, 3]
    assert mask.shape == (1, h, w, 1)
    assert torch.equal(torch.cat([c.directions for c in chunks]), rays.directions.reshape(-1, 3))


def test_synthetic_blender_rays_shape():
    r = mp.blender_rays(mp.spheric_pose(1.0))
    assert r.origins.shape == (800, 800, 3) and r.radii.dtype == np.float32
    assert abs(float(np.linalg.norm(r.origins[0, 0])) - 4.0) < 1e-5
    assert abs(float(r.radii.mean()) - 5.196e-4) < 2e-6                   # SURVEY.md §8a a0
    n = np.linalg.norm(r.directions, axis=-1)
    assert n.min() >= 1.0 - 1e-6 and n.max() < 1.13
    ms = mp.random_ray_batch(64, seed=1, multiscale=True)
    assert sorted(set(ms.lossmult.flatten().tolist())) == [1.0, 4.0, 16.0, 64.0]


def test_weights_generator_is_deterministic():
    a, b = make_state_dict(5), make_state_dict(5)
    assert all(torch.equal(a[k], b[k]) for k in a)
    x = make_state_dict(0)["mlp.layers.0.0.weight"]
    assert abs(float(x.abs().max()) - (6 / (96 + 256)) ** 0.5) < 1e-3


def test_bench_reference_arm_prints_contract_json():
    """`bench.py --impl reference` (the CPU arm the driver runs first) needs no GPU and prints one JSON line
    with the contract's keys."""
    import json
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "1"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["unit"] == "rays/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port"
    assert line["e2e"]["h2d_bytes_per_step"] == 0


def test_ray_staging_is_field_major_and_contiguous():
    rays = mp.random_ray_batch(37, seed=2, multiscale=True)
    st = mp.RayStaging(rays)
    assert st.host.numel() == 13 * 37
    for got, want in zip(st.host_rays, rays):
        assert got.is_contiguous() and torch.equal(got, want.reshape(got.shape))
    other = mp.random_ray_batch(37, seed=3)
    st.fill(other)
    assert torch.equal(st.host_rays.directions, other.directions)


def test_training_and_dataset_entry_points_validate_arguments_without_gpu(lib):
    """Status codes of the training / dataset / tensor-core-linear entry points for bad arguments: every check
    happens before the first launch, so this runs without a GPU."""
    cfg = mp.MipNerf()._config()
    # workspace sizing: bounded by the chunk, zero for shapes the training step does not cover
    w4096 = lib.mipnerf_b200_train_workspace_bytes(C.byref(cfg), 4096)
    assert w4096 > 5 << 30 and lib.mipnerf_b200_train_workspace_bytes(C.byref(cfg), 10 ** 7) == w4096
    no_view = mp.MipNerf(use_viewdirs=False, mlp_net_width_condition=256)._config()
    assert lib.mipnerf_b200_train_workspace_bytes(C.byref(no_view), 64) == 0
    # forward_backward: config problems first, then NULL arguments
    rc = lib.mipnerf_b200_forward_backward(C.byref(no_view), None, None, 0, None, None, 1, 0, None, None, None, 0, 0, None,
                                           0, None)
    assert rc == _cabi.EUNSUPPORTED and b"training" in lib.mipnerf_b200_last_error()
    rc = lib.mipnerf_b200_forward_backward(C.byref(cfg), None, None, 0, None, None, 1, 0, None, None, None, 0, 0, None, 0,
                                           None)
    assert rc == _cabi.EINVAL
    # adam: step is 1-based
    assert lib.mipnerf_b200_adam_step(None, None, None, None, 0, 1e-3, 0.9, 0.999, 1e-8, 0, 1.0, None) == _cabi.EINVAL
    assert lib.mipnerf_b200_adam_step(None, None, None, None, 0, 1e-3, 0.9, 0.999, 1e-8, 1, 1.0, None) == _cabi.OK
    assert lib.mipnerf_b200_adam_step(None, None, None, None, 5, 1e-3, 0.9, 0.999, 1e-8, 1, 1.0, None) == _cabi.EINVAL
    # tensor-core linear: shapes / precision / scratch
    assert lib.mipnerf_b200_linear_tc(None, None, None, None, 0, 64, 256, 0, _cabi.BF16, None, 0, None) == _cabi.EUNSUPPORTED
    assert lib.mipnerf_b200_linear_tc(None, None, None, None, 0, 256, 256, 0, _cabi.FP32, None, 0, None) == _cabi.EINVAL
    assert lib.mipnerf_b200_linear_tc(None, None, None, None, 0, 256, 256, 0, _cabi.BF16, None, 0, None) == _cabi.EWORKSPACE
    # ray bank / distloss
    assert lib.mipnerf_b200_rays_from_pixels(None, None, None, 0, None, 0, None, None, None, None, None, None, None, None,
                                             None, None) == _cabi.EINVAL
    assert lib.mipnerf_b200_distloss(None, None, -1, 128, None, None) == _cabi.EINVAL
    assert lib.mipnerf_b200_distloss(None, None, 0, 128, None, None) == _cabi.OK


def test_public_header_is_plain_c_and_links(tmp_path):
    """include/mipnerf_b200.h is a C header (no torch / C++ types): a C99 translation unit that includes it compiles
    with -Wall -Wextra -pedantic -Werror and links against the shared library."""
    import shutil
    import subprocess
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("no gcc")
    src = tmp_path / "abi_check.c"
    src.write_text('#include "mipnerf_b200.h"\n#include <stdio.h>\n'
                   'int main(void) {\n'
                   '  mipnerf_b200_config cfg; mipnerf_b200_loss loss; mipnerf_b200_linear_grad g;\n'
                   '  (void)cfg; (void)loss; (void)g;\n'
                   '  printf("%d %d\\n", mipnerf_b200_abi_version(), MIPNERF_B200_ABI_VERSION);\n'
                   '  return mipnerf_b200_abi_version() == MIPNERF_B200_ABI_VERSION ? 0 : 1;\n}\n')
    exe = tmp_path / "abi_check"
    libdir = os.path.join(ROOT, "mipnerf_pl_b200")
    subprocess.run([gcc, "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"),
                    str(src), "-o", str(exe), "-L", libdir, "-l:libmipnerf_b200.so", f"-Wl,-rpath,{libdir}"], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True)
    assert out.returncode == 0 and out.stdout.split() == ["4", "4"], out
