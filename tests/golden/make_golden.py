"""Generate the golden fixtures in this directory FROM THE REFERENCE ITSELF.

Run in the build container only (needs /root/reference, which does not exist on the GPU box):

    python tests/golden/make_golden.py

It imports the unmodified hjxwhy/mipnerf_pl `models.mip` / `models.mip_nerf`, runs them on CPU
(fp32) on deterministic inputs, and stores inputs + outputs as small .npz files.  The tests pin
`oracle/mipnerf_oracle.py` and the CUDA kernels against these files.  Nothing from the reference's
source is copied; only its numerical outputs are recorded.

The resampler's `inds` are not returned by the reference, so they are captured by wrapping
`torch.searchsorted` while the reference's own `sorted_piecewise_constant_pdf` runs.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.abspath(os.path.join(HERE, "..", ".."))
REF = os.environ.get("MIPNERF_REFERENCE", "/root/reference")
sys.path.insert(0, REF)
sys.path.insert(1, ROOT)

from models import mip as ref_mip  # noqa: E402  (reference)
from models.mip_nerf import MipNerf as RefMipNerf  # noqa: E402  (reference)
from datasets.datasets import Rays as RefRays  # noqa: E402  (reference)

from mipnerf_pl_b200.rays import random_ray_batch  # noqa: E402  (ours: input generator only)
from mipnerf_pl_b200.weights import make_state_dict  # noqa: E402

torch.set_num_threads(8)
F32_EPS = float(torch.finfo(torch.float32).eps)


class CaptureSearchsorted:
    """Record what torch.searchsorted returns inside the reference call."""

    def __enter__(self):
        self.calls = []
        self._orig = torch.searchsorted

        def wrapped(*a, **k):
            out = self._orig(*a, **k)
            self.calls.append(out.clone())
            return out
        torch.searchsorted = wrapped
        return self

    def __exit__(self, *exc):
        torch.searchsorted = self._orig


def to_ref_rays(r):
    return RefRays(*[getattr(r, k) for k in RefRays._fields])


def rays_dict(r):
    return {f"rays_{k}": getattr(r, k).numpy() for k in r._fields}


def save(name, **arrays):
    path = os.path.join(HERE, name)
    np.savez_compressed(path, **arrays)
    print(f"{name}: {os.path.getsize(path) / 1024:.1f} KiB")


def forward_case(name, num_rays, seed, weights_kind, randomized, white_bkgd, multiscale=False, **model_kw):
    rays = random_ray_batch(num_rays, seed=seed, multiscale=multiscale)
    shape_kw = {}
    if "max_deg_point" in model_kw or "min_deg_point" in model_kw:
        shape_kw["xyz_dim"] = 6 * (model_kw.get("max_deg_point", 16) - model_kw.get("min_deg_point", 0))
    if "deg_view" in model_kw:
        shape_kw["view_dim"] = 6 * model_kw["deg_view"] + 3
    sd = make_state_dict(seed=seed, kind=weights_kind, **shape_kw)
    model = RefMipNerf(**model_kw)
    model.load_state_dict(sd)
    model.eval()
    n = model.num_samples
    extra = {}
    if randomized:
        # replay the reference's draws: torch.rand(B,N+1) at level 0 (mip.py:159), then
        # empty(B,N+1).uniform_(to=s-eps) at level 1 (mip.py:201-202), from a seeded CPU generator.
        # With density_noise > 0 each level also draws randn(B,N,1) right after its MLP (mip_nerf.py:233), i.e. the
        # generator is consumed in the order rand, randn, uniform_, randn.
        noisy = model.density_noise > 0
        torch.manual_seed(1234 + seed)
        extra["t_rand"] = torch.rand(num_rays, n + 1).numpy()
        if noisy:
            extra["density_normal_l0"] = torch.randn(num_rays, n, 1).numpy()[..., 0]
        if model.num_levels > 1:
            s = 1 / (n + 1)
            extra["u_jitter"] = torch.empty(num_rays, n + 1).uniform_(to=(s - F32_EPS)).numpy()
            if noisy:
                extra["density_normal_l1"] = torch.randn(num_rays, n, 1).numpy()[..., 0]
        torch.manual_seed(1234 + seed)
    with torch.no_grad(), CaptureSearchsorted() as cap:
        ret = model(to_ref_rays(rays), randomized, white_bkgd)
    out = dict(rays_dict(rays))
    out.update(extra)
    for lvl, (rgb, dist, acc, w, t) in enumerate(ret):
        out[f"l{lvl}_comp_rgb"], out[f"l{lvl}_distance"], out[f"l{lvl}_acc"] = rgb.numpy(), dist.numpy(), acc.numpy()
        out[f"l{lvl}_weights"], out[f"l{lvl}_t_samples"] = w.numpy(), t.numpy()
    for i, inds in enumerate(cap.calls):
        out[f"l{i + 1}_inds"] = inds.numpy()
    out["meta"] = np.array([seed, int(randomized), int(white_bkgd)], dtype=np.int64)
    save(name, **out)


def resampler_case():
    g = torch.Generator().manual_seed(7)
    b, n = 24, 128
    dists = {
        "random4": torch.rand(b, n, generator=g) ** 4,
        "near_uniform": 0.01 + 1e-6 * torch.rand(b, n, generator=g),
        "uniform": torch.full((b, n), 0.01),
        "tiny": 1e-9 * torch.rand(b, n, generator=g),           # exercises the eps padding branch
        "spiky": torch.zeros(b, n).scatter_(1, torch.randint(0, n, (b, 3), generator=g), 1.0),
        "zeros": torch.zeros(b, n),
    }
    out = {}
    base = torch.linspace(2.0, 6.0, n + 1)[None].repeat(b, 1)
    bins = base + 0.02 * torch.rand(b, n + 1, generator=g)
    bins = torch.sort(bins, dim=-1).values
    out["bins"] = bins.numpy()
    s = 1 / (n + 1)
    torch.manual_seed(99)
    jitter = torch.empty(b, n + 1).uniform_(to=(s - F32_EPS))
    out["u_jitter"] = jitter.numpy()
    for name, w in dists.items():
        out[f"{name}_weights"] = w.numpy()
        for rand in (False, True):
            tag = f"{name}_{'rand' if rand else 'det'}"
            torch.manual_seed(99)  # reference draws the same jitter again
            with CaptureSearchsorted() as cap:
                samples = ref_mip.sorted_piecewise_constant_pdf(bins.clone(), w.clone(), n + 1, rand)
            out[f"{tag}_samples"] = samples.numpy()
            out[f"{tag}_inds"] = cap.calls[0].numpy()
    # full resample_along_rays (blur + padding) on compositing-like weights
    w = torch.rand(b, n, generator=g) ** 6
    w = w / w.sum(-1, keepdim=True) * torch.rand(b, 1, generator=g)
    rays = random_ray_batch(b, seed=3)
    with CaptureSearchsorted() as cap:
        new_t, (means, covs) = ref_mip.resample_along_rays(rays.origins, rays.directions, rays.radii, bins.clone(),
                                                           w.clone(), False, "cone", True, 0.01)
    out.update({"rs_weights": w.numpy(), "rs_new_t": new_t.numpy(), "rs_means": means.numpy(),
                "rs_covs": covs.numpy(), "rs_inds": cap.calls[0].numpy()})
    out.update({f"rs_{k}": v for k, v in rays_dict(rays).items()})
    # a 64-bin histogram (config-0 sized)
    w64 = torch.rand(b, 64, generator=g) ** 3
    bins64 = torch.sort(2 + 4 * torch.rand(b, 65, generator=g), dim=-1).values
    with CaptureSearchsorted() as cap:
        s64 = ref_mip.sorted_piecewise_constant_pdf(bins64.clone(), w64.clone(), 65, False)
    out.update({"n64_weights": w64.numpy(), "n64_bins": bins64.numpy(), "n64_samples": s64.numpy(),
                "n64_inds": cap.calls[0].numpy()})
    save("resampler.npz", **out)


def stages_case():
    g = torch.Generator().manual_seed(11)
    b, n = 12, 128
    rays = random_ray_batch(b, seed=5, multiscale=True)
    out = dict(rays_dict(rays))
    # sample_along_rays: deterministic, disparity, randomized (seeded)
    t, (m, c) = ref_mip.sample_along_rays(rays.origins, rays.directions, rays.radii, n, rays.near, rays.far,
                                          False, False, "cone")
    out.update(sa_t=t.numpy(), sa_means=m.numpy(), sa_covs=c.numpy())
    t, (m, c) = ref_mip.sample_along_rays(rays.origins, rays.directions, rays.radii, n, rays.near, rays.far,
                                          False, True, "cone")
    out.update(sa_disp_t=t.numpy(), sa_disp_means=m.numpy(), sa_disp_covs=c.numpy())
    torch.manual_seed(21)
    t_rand = torch.rand(b, n + 1)
    torch.manual_seed(21)
    t, (m, c) = ref_mip.sample_along_rays(rays.origins, rays.directions, rays.radii, n, rays.near, rays.far,
                                          True, False, "cone")
    out.update(sa_rand_t_rand=t_rand.numpy(), sa_rand_t=t.numpy(), sa_rand_means=m.numpy(), sa_rand_covs=c.numpy())
    # IPE on the randomized Gaussians (+ a stress set with tiny/huge covariances) and view PE
    enc = ref_mip.integrated_pos_enc((m, c), 0, 16)
    out["ipe_enc"] = enc.numpy()
    m2 = 6 * (torch.rand(4, 16, 3, generator=g) - 0.5)   # reference IPE wants [B,N,3]
    c2 = 10 ** (-9 + 9 * torch.rand(4, 16, 3, generator=g))
    out.update(ipe2_means=m2.numpy(), ipe2_covs=c2.numpy(),
               ipe2_enc=ref_mip.integrated_pos_enc((m2, c2), 0, 16).numpy(),
               ipe2_enc_deg2_9=ref_mip.integrated_pos_enc((m2, c2), 2, 9).numpy())
    out["pe_view"] = ref_mip.pos_enc(rays.viewdirs, 0, 4, True).numpy()
    out["pe_view_noid"] = ref_mip.pos_enc(rays.viewdirs, 0, 4, False).numpy()
    # volumetric_rendering on random activations with a hard surface in some rays
    rgb = torch.rand(b, n, 3, generator=g)
    dens = 30 * torch.rand(b, n, 1, generator=g) ** 8
    dens[::3, 40:44] = 500.0
    for wb in (True, False):
        comp, dist, acc, w = ref_mip.volumetric_rendering(rgb, dens, t, rays.directions, wb)
        tag = "vr_white" if wb else "vr_black"
        out.update({f"{tag}_comp": comp.numpy(), f"{tag}_dist": dist.numpy(), f"{tag}_acc": acc.numpy(),
                    f"{tag}_weights": w.numpy()})
    out.update(vr_rgb=rgb.numpy(), vr_density=dens.numpy(), vr_t=t.numpy())
    # distloss on the white-background compositing weights
    out["distloss_value"] = np.array(float(ref_mip.distloss(w, t)), dtype=np.float64)
    out["distloss_weights"] = w.numpy()
    # MLP.forward
    model = RefMipNerf()
    model.load_state_dict(make_state_dict(seed=2))
    x = enc[:4]
    venc = ref_mip.pos_enc(rays.viewdirs[:4], 0, 4, True)
    with torch.no_grad():
        raw_rgb, raw_density = model.mlp(x, venc)
    out.update(mlp_x=x.numpy(), mlp_venc=venc.numpy(), mlp_raw_rgb=raw_rgb.numpy(),
               mlp_raw_density=raw_density.numpy())
    save("stages.npz", **out)


GRAD_STRIDE = 37  # the gradient digest keeps every 37th element of each tensor (+ norms and sums)


def training_case():
    """Loss and parameter gradients of MipNeRFSystem.training_step (models/nerf_system.py:95-111) computed by
    the reference MipNerf + reference distloss + torch autograd; Adam/MipLRDecay trajectories from
    torch.optim.Adam and the reference's utils/lr_schedule.py.  pytorch_lightning is not installed, so the
    ten lines of loss arithmetic are restated here around the reference's own modules."""
    from utils.lr_schedule import MipLRDecay as RefMipLRDecay  # reference
    out = {}
    for tag, seed, randomized, white, disable_ms in (("a", 7, False, True, False), ("b", 8, True, False, True)):
        b = 48
        rays = random_ray_batch(b, seed=seed, multiscale=True)
        g = torch.Generator().manual_seed(100 + seed)
        rgbs = torch.rand(b, 3, generator=g)
        model = RefMipNerf()
        model.load_state_dict(make_state_dict(seed=seed, kind="trained_like"))
        model.train()
        n = model.num_samples
        if randomized:
            torch.manual_seed(4321 + seed)
            out[f"{tag}_t_rand"] = torch.rand(b, n + 1).numpy()
            out[f"{tag}_u_jitter"] = torch.empty(b, n + 1).uniform_(to=(1 / (n + 1) - F32_EPS)).numpy()
            torch.manual_seed(4321 + seed)
        ret = model(to_ref_rays(rays), randomized, white)
        mask = torch.ones_like(rays.lossmult) if disable_ms else rays.lossmult
        losses, dls = [], []
        for (rgb, _, _, weights, t_samples) in ret:
            losses.append((mask * (rgb - rgbs[..., :3]) ** 2).sum() / mask.sum())
            dls.append(ref_mip.distloss(weights, t_samples))
        loss = 0.1 * (losses[0] + 0.01 * dls[0]) + losses[1] + 0.01 * dls[-1]
        loss.backward()
        out.update({f"{tag}_{k}": v for k, v in rays_dict(rays).items()})
        out[f"{tag}_rgbs"] = rgbs.numpy()
        out[f"{tag}_loss"] = np.array([float(loss)] + [float(x) for x in losses] + [float(x) for x in dls])
        out[f"{tag}_meta"] = np.array([seed, int(randomized), int(white), int(disable_ms)], dtype=np.int64)
        for name, prm in model.named_parameters():
            gr = prm.grad.reshape(-1)
            out[f"{tag}_grad_{name}"] = gr[::GRAD_STRIDE].numpy()
            out[f"{tag}_gnorm_{name}"] = np.array([float(gr.double().norm()), float(gr.double().sum())])
    # Adam + MipLRDecay: 4 steps on one tensor, lr from the reference scheduler
    g = torch.Generator().manual_seed(9)
    p = torch.nn.Parameter(torch.randn(1000, generator=g))
    grads = torch.randn(4, 1000, generator=g) * torch.tensor([1e-3, 1.0, 1e3, 1e-6])[:, None]
    opt = torch.optim.Adam([p], lr=5e-4)
    sched = RefMipLRDecay(opt, 5e-4, 5e-6, 10, 4, 0.01)
    out["adam_p0"] = p.detach().clone().numpy()
    out["adam_grads"] = grads.numpy()
    lrs, traj = [], []
    for i in range(4):
        lrs.append(opt.param_groups[0]["lr"])
        p.grad = grads[i].clone()
        opt.step()
        sched.step()
        traj.append(p.detach().clone().numpy())
    out["adam_lrs"] = np.array(lrs)
    out["adam_traj"] = np.stack(traj)
    steps = [0, 1, 10, 1249, 2500, 2501, 100000, 999999, 1000000, 1500000]
    dummy = torch.optim.SGD([torch.nn.Parameter(torch.zeros(1))], lr=1.0)
    ref_s = RefMipLRDecay(dummy, 5e-4, 5e-6, 1000000, 2500, 0.01)
    vals = []
    for st in steps:
        ref_s.last_epoch = st
        vals.append(ref_s.get_lr()[0])
    out["lr_steps"] = np.array(steps, dtype=np.int64)
    out["lr_values"] = np.array(vals, dtype=np.float64)
    nodelay = RefMipLRDecay(dummy, 1e-3, 1e-5, 100, 0, 1.0)
    vals = []
    for st in (0, 50, 100):
        nodelay.last_epoch = st
        vals.append(nodelay.get_lr()[0])
    out["lr_nodelay_values"] = np.array(vals, dtype=np.float64)
    save("training.npz", **out)


def datasets_case():
    """The reference's own loaders (datasets/datasets.py Blender + Multicam) and multi-scale converter
    (datasets/convert_blender_data.py) run on a tiny synthetic Blender-format scene; the scene is rebuilt
    bit-identically by mipnerf_pl_b200.write_synthetic_blender_scene(root, 3, 16, 16, seed=5) in the tests."""
    import json
    import tempfile
    from datasets.datasets import Blender as RefBlender, Multicam as RefMulticam  # reference
    from datasets.convert_blender_data import convert_to_nerfdata  # reference
    from mipnerf_pl_b200.datasets import write_synthetic_blender_scene  # ours: input generator only
    root = tempfile.mkdtemp()
    write_synthetic_blender_scene(root, 3, 16, 16, seed=5)
    out = {}
    for white in (True, False):
        tag = "w" if white else "k"
        ds = RefBlender(root, "train", white_bkgd=white)
        out.update({f"blender_{tag}_train_{k}": np.asarray(getattr(ds.rays, k)) for k in RefRays._fields})
        out[f"blender_{tag}_train_images"] = np.asarray(ds.images)
    dv = RefBlender(root, "val", batch_type="single_image")
    rays1, img1 = dv[0]
    rays2, img2 = dv[0]          # val ignores the index and cycles
    out.update({f"blender_val1_{k}": np.asarray(getattr(rays2, k)) for k in RefRays._fields})
    out["blender_val1_image"] = np.asarray(img2)
    out["blender_focal"] = np.array(dv.focal)
    ms_root = root + "_ms"
    convert_to_nerfdata(root, ms_root, 3)
    meta = json.load(open(os.path.join(ms_root, "metadata.json")))["train"]
    for k in ("pix2cam", "cam2world", "width", "height", "focal", "lossmult", "near", "far", "label"):
        out[f"ms_meta_{k}"] = np.array(meta[k], dtype=np.float64)
    out["ms_meta_file_path"] = np.array(meta["file_path"])
    mt = RefMulticam(ms_root, "train")
    out.update({f"ms_train_{k}": np.asarray(getattr(mt.rays, k)) for k in RefRays._fields})
    out["ms_train_images"] = np.asarray(mt.images)
    mv = RefMulticam(ms_root, "test", batch_type="single_image")
    r, im = mv[4]
    out.update({f"ms_test4_{k}": np.asarray(getattr(r, k)) for k in RefRays._fields})
    out["ms_test4_image"] = np.asarray(im)
    save("datasets.npz", **out)


def metrics_case():
    """eval_errors / calc_psnr / ssim of the reference (utils/metrics.py:44-126, 182-197) on small synthetic frames:
    a smooth image against a noisy copy (high SSIM), against an unrelated one (low SSIM), odd sizes (tile edges of the
    CUDA kernel), plus the 1-D window itself."""
    from utils import metrics as ref_metrics  # reference
    rng = np.random.RandomState(11)
    out = {}
    for tag, (h, w) in (("a", (37, 29)), ("b", (16, 48)), ("c", (50, 50))):
        yy, xx = np.meshgrid(np.linspace(0, 3, h), np.linspace(0, 2, w), indexing="ij")
        base = np.stack([0.5 + 0.4 * np.sin(3 * xx + c) * np.cos(2 * yy) for c in range(3)], -1).astype(np.float32)
        noisy = np.clip(base + rng.normal(0, 0.03, base.shape), 0, 1).astype(np.float32)
        other = rng.uniform(0, 1, base.shape).astype(np.float32)
        for name, (p_, t_) in (("near", (noisy, base)), ("far", (other, base))):
            pred, tgt = torch.from_numpy(p_)[None], torch.from_numpy(t_)[None]
            psnr, ssim = ref_metrics.eval_errors(pred, tgt)
            out[f"{tag}_{name}_pred"], out[f"{tag}_{name}_target"] = p_, t_
            out[f"{tag}_{name}_psnr"], out[f"{tag}_{name}_ssim"] = np.float32(psnr.item()), np.float32(ssim.item())
    out["window"] = ref_metrics.get_gaussian_kernel(11, 1.5).numpy()
    save("metrics.npz", **out)


def degrees_case():
    # lower encoding degrees than the default 16 / 4 (NeRF's own 10 for points; 2 for view directions): layers.0 is
    # [256,60], layers.5 [256,316], view_layers.0 [128,271]
    forward_case("forward_deg10_view2.npz", 32, seed=6, weights_kind="trained_like", randomized=False,
                 white_bkgd=True, max_deg_point=10, deg_view=2)


def density_noise_case():
    # randomized forward with the density-noise regulariser on (models/mip_nerf.py:232-233; std 1.0 is the value the
    # NeRF papers use on real scenes), CPU reference, the generator's draws replayed into the fixture
    forward_case("forward_density_noise.npz", 24, seed=5, weights_kind="trained_like", randomized=True,
                 white_bkgd=True, density_noise=1.0)


def reference_arm_case():
    # what bench.py's CPU arm computes: 96 rays of the benchmark's ray generator (seed 0), both weight sets
    for kind in ("xavier", "trained_like"):
        forward_case(f"reference_arm_{kind}.npz", 96, seed=0, weights_kind=kind, randomized=False, white_bkgd=True)


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "reference_arm":   # regenerate only reference_arm_*.npz
        reference_arm_case()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "metrics":    # regenerate only metrics.npz
        metrics_case()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "training":   # regenerate only training.npz
        training_case()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "degrees":   # regenerate only forward_deg10_view2.npz
        degrees_case()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "density_noise":   # regenerate only forward_density_noise.npz
        density_noise_case()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "datasets":   # regenerate only datasets.npz
        datasets_case()
        sys.exit(0)
    forward_case("forward_xavier.npz", 40, seed=0, weights_kind="xavier", randomized=False, white_bkgd=True)
    forward_case("forward_trained_like.npz", 40, seed=1, weights_kind="trained_like", randomized=False,
                 white_bkgd=False, multiscale=True)
    forward_case("forward_randomized.npz", 24, seed=2, weights_kind="trained_like", randomized=True,
                 white_bkgd=True)
    forward_case("forward_config0.npz", 256, seed=3, weights_kind="xavier", randomized=False, white_bkgd=True,
                 num_samples=64, num_levels=1)
    density_noise_case()
    degrees_case()
    reference_arm_case()
    resampler_case()
    stages_case()
    training_case()
    datasets_case()
    metrics_case()
    with open(os.path.join(HERE, "VERSIONS.txt"), "w") as f:
        f.write(f"torch {torch.__version__}\nnumpy {np.__version__}\nreference {REF} (hjxwhy/mipnerf_pl @ 6c07452)\n"
                f"cpu_capability {torch.backends.cpu.get_cpu_capability()}\n")
