"""Tensor-level wrappers of the C-ABI stages (one function per kernel K1..K6).

These take/return CUDA fp32 torch tensors, allocate the outputs with torch's caching
allocator and launch on torch's current stream.  They are what the renderer composes; the
parity tests call them directly with teacher-forced inputs.
"""
from __future__ import annotations

import torch

from . import _lib
from ._lib import check, load, ptr, require_device, stream_ptr


def _f32c(t: torch.Tensor | None) -> torch.Tensor | None:
    if t is None:
        return None
    if t.dtype != torch.float32:
        raise TypeError(f'expected float32 tensor, got {t.dtype}')
    return t.contiguous()


def sample_stratified(n_rays: int, n_samples: int, near: float, far: float, u: torch.Tensor | None,
                      device: torch.device) -> torch.Tensor:
    """K1 -- generate_samples (reference src/Methods/NeRF/utils.py:57-75)."""
    z = torch.empty((n_rays, n_samples), dtype=torch.float32, device=device)
    require_device(z)
    u = _f32c(u)
    if u is not None and tuple(u.shape) != (n_rays, n_samples):
        raise ValueError(f'noise shape {tuple(u.shape)} != {(n_rays, n_samples)}')
    check(load().nerf_sample_stratified(ptr(z), ptr(u), n_rays, n_samples, float(near), float(far), stream_ptr()),
          'nerf_sample_stratified')
    return z


def sample_importance(z_coarse: torch.Tensor, w_coarse: torch.Tensor, n_fine: int, u: torch.Tensor | None,
                      return_fine: bool = False):
    """K2 -- generate_samples_from_pdf + sort(cat()) (reference utils.py:78-109, Renderer.py:70)."""
    z_coarse, w_coarse, u = _f32c(z_coarse), _f32c(w_coarse), _f32c(u)
    require_device(z_coarse)
    n, nc = z_coarse.shape
    if tuple(w_coarse.shape) != (n, nc):
        raise ValueError('weights and coarse depths differ in shape')
    if u is not None and tuple(u.shape) != (n, n_fine):
        raise ValueError(f'noise shape {tuple(u.shape)} != {(n, n_fine)}')
    merged = torch.empty((n, nc + n_fine), dtype=torch.float32, device=z_coarse.device)
    fine = torch.empty((n, n_fine), dtype=torch.float32, device=z_coarse.device) if return_fine else None
    check(load().nerf_sample_importance(ptr(merged), ptr(fine), ptr(z_coarse), ptr(w_coarse), ptr(u), n, nc, n_fine,
                                        stream_ptr()), 'nerf_sample_importance')
    return (merged, fine) if return_fine else merged


def composite_forward(z: torch.Tensor, rgbsigma: torch.Tensor, dirs: torch.Tensor, background: torch.Tensor | None,
                      want_weights: bool = False):
    """K5 -- integrate_samples (reference utils.py:112-136).  rgbsigma: (n, S, 4)."""
    z, rgbsigma, dirs, background = _f32c(z), _f32c(rgbsigma), _f32c(dirs), _f32c(background)
    require_device(z)
    n, s = z.shape
    if rgbsigma.numel() != n * s * 4:
        raise ValueError('rgbsigma must hold 4 floats per sample')
    rgb = torch.empty((n, 3), dtype=torch.float32, device=z.device)
    depth = torch.empty((n, 1), dtype=torch.float32, device=z.device)
    alpha = torch.empty((n, 1), dtype=torch.float32, device=z.device)
    w = torch.empty((n, s), dtype=torch.float32, device=z.device) if want_weights else None
    check(load().nerf_composite_forward(ptr(rgb), ptr(depth), ptr(alpha), ptr(w), ptr(z), ptr(rgbsigma), ptr(dirs),
                                        ptr(background), n, s, stream_ptr()), 'nerf_composite_forward')
    return rgb, depth, alpha, w


def composite_backward(z, rgbsigma, dirs, background, g_rgb, g_depth=None, g_alpha=None, relu_mask: bool = False,
                       grad_scale: float = 1.0) -> torch.Tensor:
    """K6 -- closed-form autograd of integrate_samples (SURVEY.md A.9).  Returns (n, S, 4)."""
    z, rgbsigma, dirs, background = _f32c(z), _f32c(rgbsigma), _f32c(dirs), _f32c(background)
    g_rgb, g_depth, g_alpha = _f32c(g_rgb), _f32c(g_depth), _f32c(g_alpha)
    require_device(z)
    n, s = z.shape
    out = torch.empty((n, s, 4), dtype=torch.float32, device=z.device)
    check(load().nerf_composite_backward(ptr(out), ptr(z), ptr(rgbsigma), ptr(dirs), ptr(background), ptr(g_rgb),
                                         ptr(g_depth), ptr(g_alpha), n, s, int(relu_mask), float(grad_scale),
                                         stream_ptr()), 'nerf_composite_backward')
    return out



def loss_mse(rgb: torch.Tensor, rgb_coarse: torch.Tensor | None, alpha: torch.Tensor | None, alpha_coarse: torch.Tensor | None,
             rgb_gt: torch.Tensor, alpha_gt: torch.Tensor | None, background: torch.Tensor | None, lambda_color: float,
             lambda_alpha: float, loss_out: torch.Tensor | None = None):
    """K8 -- NeRFLoss.forward + gradient (reference src/Methods/NeRF/Loss.py:26-43).  Returns
    (loss scalar tensor, g_rgb, g_rgb_coarse | None, g_alpha | None, g_alpha_coarse | None)."""
    rgb, rgb_coarse, alpha, alpha_coarse = _f32c(rgb), _f32c(rgb_coarse), _f32c(alpha), _f32c(alpha_coarse)
    rgb_gt, alpha_gt, background = _f32c(rgb_gt), _f32c(alpha_gt), _f32c(background)
    require_device(rgb)
    n = rgb.shape[0]
    if tuple(rgb.shape) != (n, 3) or tuple(rgb_gt.shape) != (n, 3):
        raise ValueError('rgb and rgb_gt must have shape (n, 3)')
    loss = loss_out if loss_out is not None else torch.empty((), dtype=torch.float32, device=rgb.device)
    g_rgb = torch.empty_like(rgb)
    g_rgb_c = torch.empty_like(rgb_coarse) if rgb_coarse is not None else None
    with_alpha = lambda_alpha > 0 and alpha is not None
    g_alpha = torch.empty(n, dtype=torch.float32, device=rgb.device) if with_alpha else None
    g_alpha_c = torch.empty(n, dtype=torch.float32, device=rgb.device) if with_alpha and alpha_coarse is not None else None
    check(load().nerf_loss_mse(ptr(loss), ptr(g_rgb), ptr(g_rgb_c), ptr(g_alpha), ptr(g_alpha_c), ptr(rgb), ptr(rgb_coarse),
                               ptr(alpha if with_alpha else None), ptr(alpha_coarse if with_alpha else None), ptr(rgb_gt), ptr(alpha_gt),
                               ptr(background), n, float(lambda_color), float(lambda_alpha), stream_ptr()), 'nerf_loss_mse')
    return loss, g_rgb, g_rgb_c, g_alpha, g_alpha_c


def generate_rays(c2w, width: int, height: int, focal_x: float, focal_y: float, center_x: float, center_y: float,
                  pixel_ids: torch.Tensor | None, device: torch.device):
    """K0 -- View.get_rays (reference src/Datasets/utils.py:1053-1074, src/Cameras/Perspective.py:64-94) for all pixels or for
    `pixel_ids` (int64 CUDA tensor).  `c2w`: 3x4 / 4x4 camera-to-world matrix (anything numpy can read as float64).
    Returns (origin, direction, view_direction), each (n, 3) fp32."""
    import ctypes

    import numpy as np
    m = np.ascontiguousarray(np.asarray(c2w, dtype=np.float64))
    if m.shape not in ((3, 4), (4, 4)):
        raise ValueError(f'c2w must be 3x4 or 4x4, got {m.shape}')
    if pixel_ids is not None:
        if pixel_ids.dtype != torch.int64:
            raise TypeError('pixel_ids must be int64')
        pixel_ids = pixel_ids.contiguous()
        require_device(pixel_ids)
        n = pixel_ids.numel()
    else:
        n = width * height
    out = [torch.empty((n, 3), dtype=torch.float32, device=device) for _ in range(3)]
    require_device(out[0])
    check(load().nerf_generate_rays(ptr(out[0]), ptr(out[1]), ptr(out[2]), ptr(pixel_ids), n,
                                    m.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), int(width), int(height), float(focal_x),
                                    float(focal_y), float(center_x), float(center_y), stream_ptr()), 'nerf_generate_rays')
    return tuple(out)


def gather_rays(dst: dict, src: dict, ids: torch.Tensor) -> None:
    """RayBatch.__getitem__(ids) into preallocated tensors (reference src/Datasets/utils.py:598-613), one launch.
    `dst` / `src`: dicts with any of origin, direction, view_direction, rgb (n,3) and alpha (n,1) fp32 CUDA tensors."""
    if ids.dtype != torch.int64:
        raise TypeError('ids must be int64')
    ids = ids.contiguous()
    require_device(ids)
    n = ids.numel()
    args_d, args_s = [], []
    for k in ('origin', 'direction', 'view_direction', 'rgb', 'alpha'):
        d, s_ = dst.get(k), src.get(k)
        if d is None or s_ is None:
            d = s_ = None
        else:
            if d.dtype != torch.float32 or s_.dtype != torch.float32 or not d.is_contiguous() or not s_.is_contiguous():
                raise TypeError(f'gather_rays: field {k} must be contiguous float32')
            if d.shape[0] != n:
                raise ValueError(f'gather_rays: destination {k} has {d.shape[0]} rows, expected {n}')
        args_d.append(ptr(d))
        args_s.append(ptr(s_))
    check(load().nerf_gather_rays(*args_d, *args_s, ptr(ids), n, stream_ptr()), 'nerf_gather_rays')

def mlp_packed_bytes() -> int:
    return int(load().nerf_mlp_packed_bytes())


def mlp_pack(params_flat: torch.Tensor, packed: torch.Tensor | None = None, with_backward: bool = True) -> torch.Tensor:
    """fp32 flat parameters of one block -> UMMA operand images (uint8 buffer)."""
    require_device(params_flat)
    if packed is None:
        packed = torch.empty(mlp_packed_bytes(), dtype=torch.uint8, device=params_flat.device)
    check(load().nerf_mlp_pack(ptr(packed), ptr(params_flat), int(with_backward), stream_ptr()), 'nerf_mlp_pack')
    return packed


def mlp_stash_bytes(n_samples: int) -> int:
    return int(load().nerf_mlp_stash_bytes(n_samples))


def mlp_forward(packed: torch.Tensor, params_flat: torch.Tensor, origins, dirs, viewdirs, z, noise=None,
                stash: torch.Tensor | None = None) -> torch.Tensor:
    """K3 -- encoding + NeRFBlock.forward at positions origins + dirs*z; returns (n, S, 4) = (r,g,b,sigma)."""
    origins, dirs, viewdirs, z, noise = _f32c(origins), _f32c(dirs), _f32c(viewdirs), _f32c(z), _f32c(noise)
    require_device(z)
    n, s = z.shape
    out = torch.empty((n, s, 4), dtype=torch.float32, device=z.device)
    check(load().nerf_mlp_forward(ptr(out), ptr(stash), ptr(packed), ptr(params_flat), ptr(origins), ptr(dirs),
                                  ptr(viewdirs), ptr(z), ptr(noise), n, s, stream_ptr()), 'nerf_mlp_forward')
    return out


def mlp_backward_workspace_bytes(n_samples: int) -> int:
    return int(load().nerf_mlp_backward_workspace_bytes(n_samples))


def mlp_backward(grads_flat: torch.Tensor, d_rgbsigma: torch.Tensor, rgbsigma: torch.Tensor, stash: torch.Tensor,
                 workspace: torch.Tensor, packed: torch.Tensor, params_flat: torch.Tensor, n_rays: int, n_samples: int,
                 grad_scale: float = 1.0) -> None:
    """K4 -- accumulates dL/dparams of one block into grads_flat."""
    require_device(grads_flat)
    check(load().nerf_mlp_backward(ptr(grads_flat), ptr(d_rgbsigma), ptr(rgbsigma), ptr(stash), ptr(workspace), ptr(packed),
                                   ptr(params_flat), n_rays, n_samples, float(grad_scale), stream_ptr()),
          'nerf_mlp_backward')


def mlp_backward_dgrad(d_rgbsigma, rgbsigma, stash, workspace, packed, params_flat, n_rays: int, n_samples: int) -> None:
    """K4a only: fills ``workspace`` with the per-layer output gradients."""
    require_device(d_rgbsigma)
    check(load().nerf_mlp_backward_dgrad(ptr(d_rgbsigma), ptr(rgbsigma), ptr(stash), ptr(workspace), ptr(packed),
                                         ptr(params_flat), n_rays, n_samples, stream_ptr()), 'nerf_mlp_backward_dgrad')


def mlp_backward_wgrad(grads_flat, stash, workspace, n_rays: int, n_samples: int, grad_scale: float = 1.0) -> None:
    """K4b only: accumulates weight/bias gradients from the two stashes."""
    require_device(grads_flat)
    check(load().nerf_mlp_backward_wgrad(ptr(grads_flat), ptr(stash), ptr(workspace), n_rays, n_samples, float(grad_scale),
                                         stream_ptr()), 'nerf_mlp_backward_wgrad')


def selftest_umma(a: torch.Tensor, b: torch.Tensor, mode: int) -> torch.Tensor:
    """D = A @ B^T on one 128-row tile through tcgen05 (tests only)."""
    a, b = _f32c(a), _f32c(b)
    require_device(a)
    assert a.shape[0] == 128 and a.shape[1] == b.shape[1]
    out = torch.empty((128, b.shape[0]), dtype=torch.float32, device=a.device)
    check(load().nerf_selftest_umma(ptr(out), ptr(a), ptr(b), b.shape[0], a.shape[1], mode, stream_ptr()),
          'nerf_selftest_umma')
    return out


def selftest_umma2(a: torch.Tensor, b: torch.Tensor, mn_major: bool = False) -> torch.Tensor:
    """D = A @ B^T on one 256-row tile through a cta_group::2 CTA pair (tests only); ``mn_major``: operands stored
    reduction-major and read as MN-major (the weight-gradient flavour)."""
    a, b = _f32c(a), _f32c(b)
    require_device(a)
    assert a.shape[0] == 256 and a.shape[1] == b.shape[1]
    out = torch.empty((256, b.shape[0]), dtype=torch.float32, device=a.device)
    fn = load().nerf_selftest_umma2_mn if mn_major else load().nerf_selftest_umma2
    check(fn(ptr(out), ptr(a), ptr(b), b.shape[0], a.shape[1], stream_ptr()), 'nerf_selftest_umma2')
    return out
