"""Dataset loaders for the two on-disk formats the reference trains on (SURVEY.md §8f N4):

* Blender (`transforms_{split}.json` + RGBA PNGs; datasets/datasets.py:171-263) and
* multi-scale Blender (`metadata.json` written by the converter; datasets/datasets.py:86-168,
  datasets/convert_blender_data.py:40-117),

in two forms:

1. `Blender` / `Multicam`: `torch.utils.data.Dataset`s with the reference's constructor arguments and
   `__getitem__` contract ((Rays, rgb) per ray for `split='train'`, per image otherwise), rays built on the host —
   the drop-in for the reference's `DataLoader` path.
2. `DeviceRayBank`: the B200-first form.  Images live in HBM as one pixel atlas and cameras as a small table; a
   training batch is a vector of pixel ids, and `mipnerf_b200_rays_from_pixels` turns it into Rays + target RGB on
   the device.  Nothing but the random ids (or nothing at all) crosses PCIe per step, and the 52 B/ray the
   reference keeps on the host for every pixel of every image (3.3 GB for the 100-image lego train split) is never
   materialised.

`convert_blender_to_multiscale` is the converter (box-filter pyramid + metadata.json).
"""
from __future__ import annotations

import json
import os
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch
from torch.utils.data import Dataset

from .rays import Rays, Rays_keys

_RADIUS_SCALE = 2.0 / np.sqrt(12.0)


# ------------------------------------------------------------------------------------------------
# scene loading (host)
# ------------------------------------------------------------------------------------------------
def _read_png(path: str) -> np.ndarray:
    from PIL import Image
    with open(path, "rb") as f:
        return np.array(Image.open(f), dtype=np.float32) / 255.0


def _composite(image: np.ndarray, white_bkgd: bool) -> np.ndarray:
    if white_bkgd and image.shape[-1] == 4:
        image = image[..., :3] * image[..., -1:] + (1.0 - image[..., -1:])   # datasets/datasets.py:205-206
    return np.ascontiguousarray(image[..., :3])


class Scene:
    """Images + per-image pinhole cameras: `pix2cam` [n,3,3] maps (x+.5, y+.5, 1) to a camera-space direction,
    `cam2world` [n,3,4]; per-image scalars `lossmult`, `near`, `far`."""

    def __init__(self, images: List[np.ndarray], pix2cam: np.ndarray, cam2world: np.ndarray, lossmult, near, far):
        self.images = images
        self.pix2cam = np.asarray(pix2cam, dtype=np.float32).reshape(-1, 3, 3)
        self.cam2world = np.asarray(cam2world, dtype=np.float32)[:, :3, :4].copy()
        n = len(images)
        self.lossmult = np.broadcast_to(np.asarray(lossmult, dtype=np.float32), (n,)).copy()
        self.near = np.broadcast_to(np.asarray(near, dtype=np.float32), (n,)).copy()
        self.far = np.broadcast_to(np.asarray(far, dtype=np.float32), (n,)).copy()
        self.heights = np.array([im.shape[0] for im in images], dtype=np.int32)
        self.widths = np.array([im.shape[1] for im in images], dtype=np.int32)

    def __len__(self):
        return len(self.images)


def load_blender_scene(data_dir: str, split: str, white_bkgd: bool = True, factor: int = 0,
                       near: float = 2.0, far: float = 6.0) -> Scene:
    """datasets/datasets.py:183-214.  Pixel (x, y) looks along ((x - w/2 + .5)/f, -(y - h/2 + .5)/f, -1)."""
    with open(os.path.join(data_dir, f"transforms_{split}.json")) as fp:
        meta = json.load(fp)
    images, cams = [], []
    for frame in meta["frames"]:
        image = _read_png(os.path.join(data_dir, frame["file_path"] + ".png"))
        if factor == 2:
            import cv2
            image = cv2.resize(image, (image.shape[1] // 2, image.shape[0] // 2), interpolation=cv2.INTER_AREA)
        elif factor > 0:
            raise ValueError(f"Blender dataset only supports factor=0 or 2, {factor} set.")
        images.append(_composite(image, white_bkgd))
        cams.append(np.array(frame["transform_matrix"], dtype=np.float32))
    h, w = images[0].shape[:2]
    focal = 0.5 * w / np.tan(0.5 * float(meta["camera_angle_x"]))
    k_inv = np.array([[1.0 / focal, 0.0, -0.5 * w / focal], [0.0, -1.0 / focal, 0.5 * h / focal], [0.0, 0.0, -1.0]],
                     dtype=np.float32)
    scene = Scene(images, np.broadcast_to(k_inv, (len(images), 3, 3)), np.stack(cams), 1.0, near, far)
    scene.focal = focal
    return scene


def load_multicam_scene(data_dir: str, split: str, white_bkgd: bool = True) -> Scene:
    """datasets/datasets.py:98-114: metadata.json[split] with file_path / pix2cam / cam2world / lossmult / near / far."""
    with open(os.path.join(data_dir, "metadata.json")) as fp:
        meta = json.load(fp)[split]
    images = [_composite(_read_png(os.path.join(data_dir, rel)), white_bkgd) for rel in meta["file_path"]]
    return Scene(images, np.array(meta["pix2cam"]), np.array(meta["cam2world"]), np.array(meta["lossmult"]),
                 np.array(meta["near"]), np.array(meta["far"]))


def image_rays(scene: Scene, index: int) -> Rays:
    """Rays of every pixel of one image as [H, W, C] float32 arrays (datasets/datasets.py:116-168, 216-263):
    directions are NOT normalised, `radii` is the y-neighbour distance of the directions times 2/sqrt(12) (last row
    repeats the previous one)."""
    h, w = int(scene.heights[index]), int(scene.widths[index])
    xs, ys = np.meshgrid(np.arange(w, dtype=np.float32) + 0.5, np.arange(h, dtype=np.float32) + 0.5, indexing="xy")
    pix = np.stack([xs, ys, np.ones_like(xs)], axis=-1)
    cam = pix @ scene.pix2cam[index].T
    c2w = scene.cam2world[index]
    directions = np.ascontiguousarray(cam @ c2w[:3, :3].T)
    origins = np.broadcast_to(c2w[:3, 3], directions.shape).copy()
    viewdirs = directions / np.linalg.norm(directions, axis=-1, keepdims=True)
    dy = np.sqrt(np.sum((directions[:-1] - directions[1:]) ** 2, axis=-1))
    dy = np.concatenate([dy, dy[-1:]], axis=0)
    ones = np.ones_like(origins[..., :1])
    return Rays(origins, directions, viewdirs.astype(np.float32), (dy[..., None] * _RADIUS_SCALE).astype(np.float32),
                ones * scene.lossmult[index], ones * scene.near[index], ones * scene.far[index])


# ------------------------------------------------------------------------------------------------
# the reference's Dataset surface
# ------------------------------------------------------------------------------------------------
class _RayDataset(Dataset):
    """datasets/datasets.py:24-83: 'train' = every ray of every image in one flat list (`batch_type='all_images'`),
    otherwise one image per item (`'single_image'`), `val` cycling through the images with its own counter."""

    def __init__(self, scene: Scene, split: str, batch_type: str):
        self.split, self.batch_type = split, batch_type
        self.scene = scene
        self.n_examples = len(scene)
        self.it = -1
        per_image = [image_rays(scene, i) for i in range(len(scene))]
        if split == "train":
            assert batch_type == "all_images", "The batch_type can only be all_images with flatten"
            self.images = np.concatenate([im.reshape(-1, 3) for im in scene.images], axis=0)
            self.rays = Rays(*[np.concatenate([getattr(r, k).reshape(-1, getattr(r, k).shape[-1]) for r in per_image])
                               for k in Rays_keys])
        else:
            assert batch_type == "single_image", "The batch_type can only be single_image without flatten"
            self.images = scene.images
            self.rays = Rays(*[[getattr(r, k) for r in per_image] for k in Rays_keys])

    def __len__(self):
        return len(self.images)

    def __getitem__(self, index):
        if self.split == "val":
            index = (self.it + 1) % self.n_examples
            self.it += 1
        return Rays(*[getattr(self.rays, k)[index] for k in Rays_keys]), self.images[index]


class Blender(_RayDataset):
    """datasets/datasets.py:171-263, same constructor."""

    def __init__(self, data_dir, split="train", white_bkgd=True, batch_type="all_images", factor=0):
        self.near, self.far = 2, 6
        scene = load_blender_scene(data_dir, split, white_bkgd, factor, self.near, self.far)
        self.h, self.w, self.focal = int(scene.heights[0]), int(scene.widths[0]), scene.focal
        self.camtoworlds = [c for c in scene.cam2world]
        super().__init__(scene, split, batch_type)


class Multicam(_RayDataset):
    """datasets/datasets.py:86-168, same constructor."""

    def __init__(self, data_dir, split="train", white_bkgd=True, batch_type="all_images"):
        super().__init__(load_multicam_scene(data_dir, split, white_bkgd), split, batch_type)


dataset_dict = {"blender": Blender, "multi_blender": Multicam}   # datasets/__init__.py


# ------------------------------------------------------------------------------------------------
# multi-scale converter
# ------------------------------------------------------------------------------------------------
def _down2(img: np.ndarray) -> np.ndarray:
    h, w = img.shape[0] // 2, img.shape[1] // 2
    return img[:2 * h, :2 * w].reshape(h, 2, w, 2, -1).mean(axis=(1, 3))


def convert_blender_to_multiscale(basedir: str, newdir: str, n_down: int = 4, splits=("train", "val", "test")):
    """datasets/convert_blender_data.py:40-117: every image at n_down box-filtered scales (focal / 2^j,
    lossmult 4^j) + metadata.json with the per-image pix2cam."""
    from PIL import Image
    os.makedirs(newdir, exist_ok=True)
    big = {}
    for split in splits:
        with open(os.path.join(basedir, f"transforms_{split}.json")) as fp:
            meta = json.load(fp)
        imgdir = f"images_{split}"
        os.makedirs(os.path.join(newdir, imgdir), exist_ok=True)
        out = {k: [] for k in ("file_path", "cam2world", "width", "height", "focal", "label", "near", "far", "lossmult")}
        focal = None
        for i, frame in enumerate(meta["frames"]):
            img = _read_png(os.path.join(basedir, frame["file_path"] + ".png"))
            if focal is None:
                focal = 0.5 * img.shape[1] / np.tan(0.5 * float(meta["camera_angle_x"]))
            for j in range(n_down):
                rel = f"{imgdir}/{i:03d}_d{j}.png"
                Image.fromarray(np.uint8(img * 255)).save(os.path.join(newdir, rel))
                out["file_path"].append(rel)
                out["cam2world"].append(np.asarray(frame["transform_matrix"]).tolist())
                out["width"].append(img.shape[1])
                out["height"].append(img.shape[0])
                out["focal"].append(focal / 2 ** j)
                out["label"].append(j)
                out["near"].append(2.0)
                out["far"].append(6.0)
                out["lossmult"].append(4.0 ** j)
                img = _down2(img)
        f = np.array(out["focal"], dtype=np.float64)
        cx, cy = np.array(out["width"]) * 0.5, np.array(out["height"]) * 0.5
        zero, one = np.zeros_like(f), np.ones_like(f)
        k_inv = np.array([[one / f, zero, -cx / f], [zero, -one / f, cy / f], [zero, zero, -one]])
        out["pix2cam"] = np.moveaxis(k_inv, -1, 0).tolist()
        big[split] = out
    with open(os.path.join(newdir, "metadata.json"), "w") as fp:
        json.dump(big, fp, ensure_ascii=False, indent=4)


# ------------------------------------------------------------------------------------------------
# device-resident form
# ------------------------------------------------------------------------------------------------
CAM_TABLE_WIDTH = 24  # pix2cam (9, row-major) | cam2world [3,4] (12, row-major) | lossmult | near | far


class DeviceRayBank:
    """All training pixels of a scene in HBM: `atlas` [P,3] target colours, `cam_table` [n,24], `offsets` [n+1]
    (first atlas row of each image), `widths` [n].  `rays(pixel_ids)` / `sample(batch)` produce (Rays, rgb) on the
    device with one kernel launch; there is no per-ray host data."""

    def __init__(self, scene: Scene, device="cuda"):
        dev = torch.device(device)
        if dev.type != "cuda":
            raise RuntimeError("DeviceRayBank keeps the scene in HBM; use Blender / Multicam for host rays")
        self.device = dev
        n = len(scene)
        table = np.concatenate([scene.pix2cam.reshape(n, 9), scene.cam2world.reshape(n, 12), scene.lossmult[:, None],
                                scene.near[:, None], scene.far[:, None]], axis=1).astype(np.float32)
        sizes = scene.heights.astype(np.int64) * scene.widths.astype(np.int64)
        offsets = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
        self.num_pixels = int(offsets[-1])
        self.num_images = n
        self.cam_table = torch.from_numpy(table).to(dev)
        self.offsets = torch.from_numpy(offsets).to(dev)
        self.widths = torch.from_numpy(scene.widths.astype(np.int32)).to(dev)
        self.atlas = torch.cat([torch.from_numpy(im.reshape(-1, 3)) for im in scene.images]).to(dev)

    def rays(self, pixel_ids: torch.Tensor) -> Tuple[Rays, torch.Tensor]:
        """pixel_ids: int64 [B] atlas rows (image-major, then row-major pixels) -> (Rays [B,*], rgb [B,3])."""
        from . import _cabi
        from .ops import _stream
        ids = pixel_ids.to(device=self.device, dtype=torch.int64).contiguous()
        b = ids.numel()
        mk = lambda c: torch.empty(b, c, device=self.device)  # noqa: E731
        o, d, v, rad, lm, nr, fr, rgb = mk(3), mk(3), mk(3), mk(1), mk(1), mk(1), mk(1), mk(3)
        with torch.cuda.device(self.device):
            _cabi.check(_cabi.lib().mipnerf_b200_rays_from_pixels(
                self.cam_table.data_ptr(), self.offsets.data_ptr(), self.widths.data_ptr(), self.num_images,
                ids.data_ptr(), b, self.atlas.data_ptr(), o.data_ptr(), d.data_ptr(), v.data_ptr(), rad.data_ptr(),
                lm.data_ptr(), nr.data_ptr(), fr.data_ptr(), rgb.data_ptr(), _stream(self.device)), "rays_from_pixels")
        return Rays(o, d, v, rad, lm, nr, fr), rgb

    def sample(self, batch_size: int, generator: Optional[torch.Generator] = None) -> Tuple[Rays, torch.Tensor]:
        """A uniformly random training batch over all pixels of all images (what shuffle=True over the flattened
        'all_images' list gives the reference, datasets/datasets.py:38-44 + models/nerf_system.py:78-83)."""
        ids = torch.randint(0, self.num_pixels, (batch_size,), device=self.device, generator=generator)
        return self.rays(ids)

    def sample_philox(self, rng_state: torch.Tensor, batch_size: int, ray_base: int = 0, out=None):
        """A uniformly random batch drawn by ONE kernel from the Philox state `rng_state` (int64 [2] on this device: seed,
        offset, read when the kernel runs -- so a CUDA graph replays it with fresh ids once the offset moves).
        Returns (Rays, rgb, pixel_ids); `out` = such a triple to write into.  `philox_pixel_ids` recomputes the ids."""
        from . import _cabi
        from .ops import _stream
        if out is None:
            mk = lambda c: torch.empty(batch_size, c, device=self.device)  # noqa: E731
            out = (Rays(mk(3), mk(3), mk(3), mk(1), mk(1), mk(1), mk(1)), mk(3),
                   torch.empty(batch_size, dtype=torch.int64, device=self.device))
        r, rgb, ids = out
        with torch.cuda.device(self.device):
            _cabi.check(_cabi.lib().mipnerf_b200_sample_pixels(
                self.cam_table.data_ptr(), self.offsets.data_ptr(), self.widths.data_ptr(), self.num_images,
                self.num_pixels, rng_state.data_ptr(), int(ray_base), batch_size, self.atlas.data_ptr(), ids.data_ptr(),
                *[f.data_ptr() for f in r], rgb.data_ptr(), _stream(self.device)), "sample_pixels")
        return out


def philox_pixel_ids(seed: int, offset: int, count: int, num_pixels: int, ray_base: int = 0) -> np.ndarray:
    """Host mirror of mipnerf_b200_sample_pixels' ids: Philox4x32-10 (the generator of the in-kernel draws,
    mipnerf_b200_philox_uniform) on counter (ray_base + i, 64 << 24, offset), key (seed, offset), first output word x;
    id = (x * num_pixels) >> 32."""
    seed &= (1 << 64) - 1
    offset &= (1 << 64) - 1
    g = np.arange(ray_base, ray_base + count, dtype=np.uint64)
    x = philox4x32_10_first(g & 0xFFFFFFFF, g >> np.uint64(32), 64 << 24, offset & 0xFFFFFFFF,
                            seed & 0xFFFFFFFF, (seed >> 32) ^ (offset >> 32))
    return ((x.astype(np.uint64) * np.uint64(num_pixels)) >> np.uint64(32)).astype(np.int64)


def philox4x32_10_first(c0, c1, c2, c3, k0, k1) -> np.ndarray:
    """First output word of Philox4x32-10 (ray_math.cuh), vectorised over the counter words."""
    m = np.uint64(0xFFFFFFFF)
    n = np.broadcast(c0, c1, c2, c3).shape
    c = [np.broadcast_to(np.asarray(v, dtype=np.uint64), n).copy() for v in (c0, c1, c2, c3)]
    k0, k1 = np.uint64(k0), np.uint64(k1)
    for _ in range(10):
        p0, p1 = np.uint64(0xD2511F53) * c[0], np.uint64(0xCD9E8D57) * c[2]
        hi0, lo0, hi1, lo1 = p0 >> np.uint64(32), p0 & m, p1 >> np.uint64(32), p1 & m
        c = [hi1 ^ c[1] ^ k0, lo1, hi0 ^ c[3] ^ k1, lo0]
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & m, (k1 + np.uint64(0xBB67AE85)) & m
    return c[0].astype(np.uint32)


def write_synthetic_blender_scene(root: str, n_images: int = 3, height: int = 16, width: int = 12, seed: int = 0,
                                  splits: Sequence[str] = ("train", "val", "test")) -> None:
    """A tiny Blender-format scene (random RGBA PNGs, poses on a sphere) for tests and smoke runs: no dataset is
    reachable offline."""
    from PIL import Image
    from .rays import spheric_pose
    rng = np.random.RandomState(seed)
    for split in splits:
        os.makedirs(os.path.join(root, split), exist_ok=True)
        frames = []
        for i in range(n_images):
            rgba = rng.randint(0, 256, size=(height, width, 4), dtype=np.uint8)
            Image.fromarray(rgba, mode="RGBA").save(os.path.join(root, split, f"r_{i}.png"))
            pose = np.eye(4, dtype=np.float64)
            pose[:3, :4] = spheric_pose(float(rng.uniform(0, 2 * np.pi)))
            frames.append({"file_path": f"./{split}/r_{i}", "transform_matrix": pose.tolist()})
        with open(os.path.join(root, f"transforms_{split}.json"), "w") as fp:
            json.dump({"camera_angle_x": 0.6911112070083618, "frames": frames}, fp)
