"""Config E of BASELINE.json: sample-count stress sweep for the HBM-bound stages (K1, K2, K5, K6).

65,536-ray batch, (Nc, Nf) in {(64,64), (64,128), (64,192), (128,256), (128,384)}; inputs as SURVEY.md 8(d):
sigma ~ Exp(1) * Bernoulli(0.5), colour ~ U[0,1], z sorted U[2,6], seed 0.  Every launch is timed alone with CUDA
events on the launching stream after an L2 flush (a 512 MB fill followed by a 512 MB read), median of `iters`; the achieved figure is the
ALGORITHMIC bytes of SURVEY.md 8(d) / DESIGN.md divided by that time.

    python tools/stress_sweep.py [--json] [--rays 65536] [--iters 7] [--profile]   (--profile: one launch each, for ncu)
"""
from __future__ import annotations

import argparse
import json
import os
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from nerficg_b200 import _lib, ops  # noqa: E402

if os.environ.get('NERF_B200_LIB'):  # development: time another build of the library
    _lib.LIB_PATH = Path(os.environ['NERF_B200_LIB']).resolve()

SWEEP = ((64, 64), (64, 128), (64, 192), (128, 256), (128, 384))


def algorithmic_bytes(n: int, nc: int, nf: int) -> dict:
    s = nc + nf
    return {
        'K1_stratified': n * nc * 8,                                  # U read + z written
        'K2_importance': n * (4 * nc + 4 * nc + 4 * nf + 4 * s),     # z_c, w_c, U read; merged z written
        'K5_composite_fwd': n * (20 * s + 32),                        # sigma+rgb+z per sample; d in, rgb/depth/alpha out
        'K5_composite_fwd_w': n * (24 * nc + 32),                     # coarse pass: + weights written
        'K6_composite_bwd': n * (36 * s + 48),                        # 20 read + 16 written per sample
    }


def run(n_rays: int = 65536, iters: int = 7, profile: bool = False, device: str = 'cuda:0') -> list[dict]:
    dev = torch.device(device)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    flush_rd = torch.zeros(128 << 20, dtype=torch.int32, device=dev)   # 512 MB read back after the fill (see timed())
    g = torch.Generator(device=dev).manual_seed(0)
    dirs = torch.nn.functional.normalize(torch.randn(n_rays, 3, generator=g, device=dev), dim=-1) * 1.05
    bg = torch.ones(3, device=dev)
    g_rgb = torch.randn(n_rays, 3, generator=g, device=dev)
    rows = []

    def timed(fn) -> float:
        ts = []
        for _ in range(1 if profile else iters + 2):
            # flush L2: write 512 MB, then READ 512 MB so that the cache is left full of clean lines -- after a pure
            # write flush the timed kernel pays for the write-back of the flush's dirty lines (measured: 5-20 us
            # kernels lost up to half of their bandwidth to it)
            flush.fill_(1)
            flush_rd.sum()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        ts = sorted(ts[2:] if not profile else ts)
        return ts[len(ts) // 2]

    # K0 (SURVEY.md 8(f) rank 1): all rays of one 800x800 view (36 B written per ray) and a 4096-ray batch gathered from a
    # 64 M-ray-sized pool slice (52 B read + 52 B written per ray)
    import numpy as np
    c2w = np.eye(4)
    c2w[:3, 3] = (0.0, -4.0, 0.5)
    n_img = 800 * 800
    t_gen = timed(lambda: ops.generate_rays(c2w, 800, 800, 1111.11, 1111.11, 400.0, 400.0, None, dev))
    pool = {k: torch.rand(4_000_000, 3, generator=g, device=dev) for k in ('origin', 'direction', 'view_direction', 'rgb')}
    pool['alpha'] = torch.rand(4_000_000, 1, generator=g, device=dev)
    ids = torch.randint(0, 4_000_000, (4096,), generator=g, device=dev)
    dst = {k: torch.empty((4096,) + tuple(t.shape[1:]), device=dev) for k, t in pool.items()}
    t_gat = timed(lambda: ops.gather_rays(dst, pool, ids))
    rows.append({'n_rays': n_img, 'n_coarse': 0, 'n_fine': 0, 'kernels': {
        'K0_generate_rays_800x800': {'us': round(1e3 * t_gen, 2), 'bytes': 36 * n_img, 'gbs': round(36 * n_img / t_gen / 1e6, 1)},
        'K0_gather_4096_rays': {'us': round(1e3 * t_gat, 2), 'bytes': 104 * 4096, 'gbs': round(104 * 4096 / t_gat / 1e6, 1)}}})
    del pool
    for nc, nf in SWEEP:
        s = nc + nf
        u_c = torch.rand(n_rays, nc, generator=g, device=dev)
        u_f = torch.rand(n_rays, nf, generator=g, device=dev)
        z = torch.sort(2 + 4 * torch.rand(n_rays, s, generator=g, device=dev), dim=-1).values
        sigma = torch.empty(n_rays, s, device=dev).exponential_(1.0, generator=g) * (torch.rand(n_rays, s, generator=g, device=dev) < 0.5)
        rs = torch.cat((torch.rand(n_rays, s, 3, generator=g, device=dev), sigma[..., None]), dim=-1).contiguous()
        z_c = ops.sample_stratified(n_rays, nc, 2.0, 6.0, u_c, dev)
        rs_c = rs[:, :nc].contiguous()
        _, _, _, w_c = ops.composite_forward(z_c, rs_c, dirs, bg, True)
        t = {
            'K1_stratified': timed(lambda: ops.sample_stratified(n_rays, nc, 2.0, 6.0, u_c, dev)),
            'K5_composite_fwd_w': timed(lambda: ops.composite_forward(z_c, rs_c, dirs, bg, True)),
            'K2_importance': timed(lambda: ops.sample_importance(z_c, w_c, nf, u_f)),
            'K5_composite_fwd': timed(lambda: ops.composite_forward(z, rs, dirs, bg)),
            'K6_composite_bwd': timed(lambda: ops.composite_backward(z, rs, dirs, bg, g_rgb, None, None, True, 1024.0)),
        }
        by = algorithmic_bytes(n_rays, nc, nf)
        rows.append({'n_rays': n_rays, 'n_coarse': nc, 'n_fine': nf,
                     'kernels': {k: {'us': round(1e3 * ms, 2), 'bytes': by[k], 'gbs': round(by[k] / ms / 1e6, 1)} for k, ms in t.items()}})
    return rows


if __name__ == '__main__':
    ap = argparse.ArgumentParser()
    ap.add_argument('--rays', type=int, default=65536)
    ap.add_argument('--iters', type=int, default=7)
    ap.add_argument('--json', action='store_true')
    ap.add_argument('--profile', action='store_true')
    a = ap.parse_args()
    out = run(a.rays, a.iters, a.profile)
    if a.json:
        print(json.dumps(out))
    else:
        for r in out:
            print(f"Nc={r['n_coarse']:3d} Nf={r['n_fine']:3d}: " + '  '.join(f"{k} {v['us']:.1f}us {v['gbs']:.0f}GB/s" for k, v in r['kernels'].items()))
