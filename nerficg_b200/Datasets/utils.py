"""Ray/data model of the NeRF path (reference src/Datasets/utils.py: RayBatch :536-670, RayCollection
:673-690, View.get_rays :1053-1074, apply_background_color :185-189).  Field names and semantics are the
reference's; everything unrelated to the vanilla-NeRF path (point clouds, flow IO, pose PCA) is absent."""
from __future__ import annotations

from dataclasses import dataclass, fields

import numpy as np
import torch

from .. import Framework
from ..Cameras.Perspective import PerspectiveCamera


@dataclass(frozen=True)
class RayBatch:
    """Per-ray tensors, all (n, C) with identical n, dtype and device."""
    origin: torch.Tensor
    direction: torch.Tensor
    view_direction: torch.Tensor | None = None
    rgb: torch.Tensor | None = None
    alpha: torch.Tensor | None = None
    depth: torch.Tensor | None = None
    timestamp: torch.Tensor | None = None
    _skip_post_init: bool = False

    _FIELDS = ('origin', 'direction', 'view_direction', 'rgb', 'alpha', 'depth', 'timestamp')

    def __post_init__(self):
        if self._skip_post_init:
            return
        n, dtype, device = self.origin.shape[0], self.origin.dtype, self.origin.device
        for member in fields(self):
            value = getattr(self, member.name)
            if isinstance(value, torch.Tensor):
                if value.shape[0] != n:
                    raise Framework.DatasetError(f'{member.name} has {value.shape[0]} rays, origin has {n}')
                if value.dtype != dtype:
                    raise Framework.DatasetError(f'{member.name} is {value.dtype}, origin is {dtype}')
                if value.device != device:
                    raise Framework.DatasetError(f'{member.name} is on {value.device}, origin is on {device}')

    def __len__(self) -> int:
        return self.origin.shape[0]

    @property
    def dtype(self) -> torch.dtype:
        return self.origin.dtype

    @property
    def device(self) -> torch.device:
        return self.origin.device

    def _map(self, fn) -> 'RayBatch':
        return RayBatch(**{k: (None if getattr(self, k) is None else fn(getattr(self, k))) for k in self._FIELDS},
                        _skip_post_init=True)

    def __getitem__(self, idx) -> 'RayBatch':
        if idx is Ellipsis or (isinstance(idx, slice) and idx == slice(None)):
            return self
        if isinstance(idx, int):
            idx = slice(idx, idx + 1)
        if isinstance(idx, torch.Tensor) and idx.dtype == torch.int64 and idx.dim() == 1 and idx.is_cuda and self.origin.is_cuda:
            return self._gather(idx)
        return self._map(lambda t: t[idx])

    _GATHERED = ('origin', 'direction', 'view_direction', 'rgb', 'alpha')

    def _gather(self, ids: torch.Tensor) -> 'RayBatch':
        """Index-tensor selection through ONE `nerf_gather_rays` launch for the five fields of the training batch
        (reference RayBatch.__getitem__, Datasets/utils.py:598-613, is one torch gather per field).  A field that requires
        grad, while grad is enabled, is gathered by torch indexing so that gradients flow back into it."""
        from .. import ops
        n = ids.numel()
        src, dst, out = {}, {}, {}
        grad_enabled = torch.is_grad_enabled()
        for k in self._FIELDS:
            t = getattr(self, k)
            if t is None:
                out[k] = None
            elif k in self._GATHERED and t.dtype == torch.float32 and t.is_contiguous() and t.dim() == 2 and \
                    t.shape[1] == (1 if k == 'alpha' else 3) and not (grad_enabled and t.requires_grad):
                src[k] = t
                dst[k] = out[k] = torch.empty((n, t.shape[1]), dtype=torch.float32, device=t.device)
            else:
                out[k] = t[ids]
        if src:
            ops.gather_rays(dst, src, ids)
        return RayBatch(**out, _skip_post_init=True)

    def to(self, dtype: torch.dtype = None, device: torch.device = None, non_blocking: bool = False) -> 'RayBatch':
        if (dtype is None or dtype == self.dtype) and (device is None or torch.device(device) == self.device):
            return self
        return self._map(lambda t: t.to(dtype=dtype, device=device, non_blocking=non_blocking))

    def cpu(self) -> 'RayBatch':
        return self.to(device=torch.device('cpu'))

    def cuda(self, non_blocking: bool = False) -> 'RayBatch':
        return self.to(device=Framework.config.GLOBAL.DEFAULT_DEVICE, non_blocking=non_blocking)

    def split(self, chunk_size: int) -> list['RayBatch']:
        return [self[i:i + chunk_size] for i in range(0, len(self), chunk_size)]

    @classmethod
    def cat(cls, batches: list['RayBatch']) -> 'RayBatch':
        if not batches:
            raise Framework.DatasetError('no RayBatch instances to concatenate')
        out = {}
        for k in cls._FIELDS:
            present = [getattr(b, k) is not None for b in batches]
            if any(present) and not all(present):
                raise Framework.DatasetError(f'RayBatch field "{k}" is not present in some batches')
            out[k] = torch.cat([getattr(b, k) for b in batches], dim=0) if all(present) else None
        return cls(**out, _skip_post_init=True)


@dataclass(frozen=True)
class RayCollection:
    """All rays of a subset with one slice per view."""
    rays: RayBatch
    camera_slices: list

    def __len__(self) -> int:
        return len(self.rays)

    def __getitem__(self, index: int) -> RayBatch:
        return self.rays[self.camera_slices[index]]

    @property
    def all_rays(self) -> RayBatch:
        return self.rays


def apply_background_color(raw_rgb: torch.Tensor, alpha: torch.Tensor, background_color: torch.Tensor,
                           is_chw: bool = True) -> torch.Tensor:
    """clamp(lerp(bg, rgb, alpha), 0, 1)."""
    if is_chw:
        background_color = background_color[:, None, None]
    return torch.lerp(background_color.to(raw_rgb.device).expand_as(raw_rgb), raw_rgb, alpha).clamp(0, 1)


class View:
    """A posed camera with optional image annotations (rgb 3xHxW, alpha 1xHxW, depth 1xHxW).

    ``c2w`` is a 4x4 (or 3x4) camera-to-world matrix whose rotation columns are the camera's x (right),
    y (down) and z (forward) axes in world space."""

    def __init__(self, camera: PerspectiveCamera, c2w: np.ndarray | torch.Tensor, rgb: torch.Tensor | None = None,
                 alpha: torch.Tensor | None = None, depth: torch.Tensor | None = None, timestamp: float = 0.0,
                 frame_idx: int = 0) -> None:
        self.camera = camera
        self.c2w = torch.as_tensor(np.asarray(c2w), dtype=torch.float32)
        self.rgb, self.alpha, self.depth = rgb, alpha, depth
        self.timestamp = timestamp
        self.frame_idx = frame_idx

    @property
    def position(self) -> torch.Tensor:
        return self.c2w[:3, 3]

    @property
    def rotation(self) -> torch.Tensor:
        return self.c2w[:3, :3]

    def get_rays(self, pixel_ids: torch.Tensor | None = None) -> RayBatch:
        """Rays of every pixel (row-major) -- or of `pixel_ids` -- on the default CUDA device, generated by K0
        (`nerf_generate_rays`; reference View.get_rays, Datasets/utils.py:1053-1074)."""
        from .. import ops
        device = Framework.config.GLOBAL.DEFAULT_DEVICE
        cam = self.camera
        if pixel_ids is not None:
            pixel_ids = pixel_ids.to(device=device, dtype=torch.int64)
        origin, direction, view_direction = ops.generate_rays(self.c2w.double().numpy(), cam.width, cam.height, cam.focal_x, cam.focal_y,
                                                              cam.center_x, cam.center_y, pixel_ids, device)
        n = direction.shape[0]

        def flat(name):
            img = getattr(self, name)
            if img is None:
                return None
            # the (H*W, C) device copy is made once per view and kept: re-uploading the whole image every training
            # iteration was 10 MB of H2D per step at 800x800 (the sampled rows are then one device gather)
            cache = self.__dict__.setdefault('_flat_device_cache', {})
            hit = cache.get(name)
            if hit is None or hit[0] is not img or hit[1].device != torch.device(device):
                hit = cache[name] = (img, img.to(device).permute(1, 2, 0).reshape(cam.width * cam.height, -1).contiguous())
            return hit[1] if pixel_ids is None else hit[1][pixel_ids]
        ts = torch.full((n, 1), float(self.timestamp), dtype=torch.float32, device=device)
        return RayBatch(origin=origin, direction=direction, view_direction=view_direction,
                        rgb=flat('rgb'), alpha=flat('alpha'), depth=flat('depth'), timestamp=ts)
