"""Timing of K4r (nerf_mlp_backward_rays) against block-mode K4c at the same sample count, and of render_rays forward +
backward with and without ray gradients.

    python tools/ray_grad_timing.py [--rays 4096] [--coarse 64] [--fine 128] [--iters 20]

K4r / K4c: CUDA events around each launch for the fine pass of `--rays` rays at `--coarse` + `--fine` samples (4096 x 192 =
786,432 samples by default), the two kernels alternating launch by launch in the same run, with L2 overwritten (a 256 MB
memset, twice the 126 MB L2) before every launch.  Both read the real gradient workspace, filled by the training forward
and dgrad of those samples.  Reports the medians and the bytes each kernel must move (computed from shapes) over its time.
render_rays: wall time of forward + backward of `--rays` rays at `--coarse` + `--fine` samples, ended by a device
synchronise, median of `--iters`, in three modes: parameters only, parameters + rays, rays only with a frozen model.
The card's name, power limit and max SM clock are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import torch  # noqa: E402

DEV = 'cuda:0'


def card() -> dict:
    r = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                       capture_output=True, text=True)
    return {'device': torch.cuda.get_device_name(0), 'nvidia_smi': r.stdout.strip()}


def panel_bytes(n: int) -> int:
    return (n + 127) // 128 * (4 + 4 + 2) * 128 * 128      # the D0, D5 and DC0 panels of every tile


def k4c_bytes(n: int) -> int:
    return panel_bytes(n) + n * 3 * 4 * 4                  # + positions, directions read, two gradients written


def k4r_bytes(n_rays: int, s: int) -> int:
    n = n_rays * s
    # + z, rgbsigma and d_rgbsigma per sample (the float4s share 32-byte sectors, so both arrays are read whole),
    # origins, dirs, viewdirs read and three accumulators read and written per ray, the per-tile scratch written and read
    return panel_bytes(n) + n * (4 + 16 + 16) + n_rays * 9 * 4 * 3 + (n + 127) // 128 * 2 * 9 * 4 * 2


def median(xs):
    return sorted(xs)[len(xs) // 2]


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument('--rays', type=int, default=4096)
    ap.add_argument('--coarse', type=int, default=64)
    ap.add_argument('--fine', type=int, default=128)
    ap.add_argument('--iters', type=int, default=20)
    args = ap.parse_args()
    from nerficg_b200 import Framework, ops
    from nerficg_b200.Cameras import PerspectiveCamera, SharedCameraSettings
    from nerficg_b200.Datasets import RayBatch
    from nerficg_b200.Methods.NeRF.Model import NeRFBlock
    from nerficg_b200.Methods.NeRF.Renderer import NeRFRayRenderingComponent
    Framework.setup(None, {'GLOBAL.LOG_LEVEL': 0})
    torch.manual_seed(0)
    coarse = NeRFBlock(8, 1, 256, 10, 4, True, [5], 'relu').to(DEV)
    fine = NeRFBlock(8, 1, 256, 10, 4, True, [5], 'relu').to(DEV)
    res = {'card': card()}

    # ---- K4r and K4c alone, alternating ----
    n_rays, s = args.rays, args.coarse + args.fine
    n = n_rays * s
    flat = fine.flat_params
    packed = ops.mlp_pack(flat)
    o = torch.nn.functional.normalize(torch.randn(n_rays, 3, device=DEV), dim=-1) * 4
    d = -o / 4 + 0.1 * torch.randn(n_rays, 3, device=DEV)
    v = torch.nn.functional.normalize(d, dim=-1)
    z = torch.sort(torch.rand(n_rays, s, device=DEV) * 4 + 2, dim=-1).values
    stash = torch.empty(ops.mlp_stash_bytes(n), dtype=torch.uint8, device=DEV)
    rs = ops.mlp_forward(packed, flat, o, d, v, z, None, stash)
    d_rs = torch.randn(n, 4, device=DEV) * 10
    ws = torch.empty(ops.mlp_backward_workspace_bytes(n), dtype=torch.uint8, device=DEV)
    ops.mlp_backward_dgrad(d_rs, rs, stash, ws, packed, flat, n_rays, s)
    pts = (o[:, None] + d[:, None] * z[..., None]).reshape(n, 3)
    vs = v[:, None].expand(-1, s, -1).reshape(n, 3).contiguous()
    acc = [torch.zeros(n_rays, 3, device=DEV) for _ in range(3)]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=DEV)
    launches = {'k4r': lambda: ops.mlp_backward_rays(*acc, ws, flat, o, d, v, z, rs, d_rs),
                'k4c': lambda: ops.mlp_backward_inputs(ws, flat, pts, vs, n)}
    times = {k: [] for k in launches}
    for i in range(args.iters + 3):
        for k, fn in launches.items():
            flush.fill_(i & 255)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            if i >= 3:
                times[k].append(a.elapsed_time(b) * 1e-3)
    for k, nbytes in (('k4r', k4r_bytes(n_rays, s)), ('k4c', k4c_bytes(n))):
        t = median(times[k])
        res[k] = {'samples': n, 'median_s': t, 'min_s': min(times[k]), 'max_s': max(times[k]), 'bytes': nbytes,
                  'bytes_per_s': nbytes / t, 'l2': 'overwritten before every launch'}
    res['k4r']['rays'] = n_rays
    res['k4r_over_k4c'] = res['k4r']['median_s'] / res['k4c']['median_s']
    del stash, ws, rs, d_rs, pts, vs, flush

    # ---- render_rays forward + backward ----
    camera = PerspectiveCamera(shared_settings=SharedCameraSettings(torch.ones(3), 2.0, 6.0), width=100, height=100,
                               focal_x=138.889, focal_y=138.889)
    comp = NeRFRayRenderingComponent(coarse, fine)
    target = torch.rand(n_rays, 3, device=DEV)
    for mode, params_grad, rays_grad in (('params', True, False), ('params+rays', True, True), ('rays_frozen_model', False, True)):
        for blk in (coarse, fine):
            blk.requires_grad_(params_grad)
        walls = []
        for i in range(args.iters + 2):
            coarse.zero_grad(set_to_none=True)
            fine.zero_grad(set_to_none=True)
            leaves = [t.clone().requires_grad_(rays_grad) for t in (o, d, v)]
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = comp(RayBatch(origin=leaves[0], direction=leaves[1], view_direction=leaves[2]), camera, 8192,
                       args.coarse, args.fine, True, 0.0)
            (((out['rgb'] - target) ** 2).mean() + ((out['rgb_coarse'] - target) ** 2).mean()).backward()
            torch.cuda.synchronize()
            if i >= 2:
                walls.append(time.perf_counter() - t0)
        res[f'render_fwd_bwd_{mode}'] = {'rays': n_rays, 'samples': f'{args.coarse}+{args.fine}', 'median_s': median(walls),
                                         'min_s': min(walls), 'max_s': max(walls)}
    print(json.dumps(res))


if __name__ == '__main__':
    main()
