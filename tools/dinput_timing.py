"""Timing of K4c (nerf_mlp_backward_inputs) and of NeRFBlock.forward + backward with input gradients.

    python tools/dinput_timing.py [--samples 786432] [--iters 20] [--block-points 1000000]

K4c: CUDA events around each launch at `--samples` samples, with L2 overwritten (a 256 MB memset, twice the 126 MB L2)
before every launch; the gradient workspace is the real one, filled by the training forward + dgrad.  Reports the median
time, the bytes the kernel must move (computed from shapes: the D0, D5 and DC0 panels of every tile, the positions and
directions it reads and the two gradients it writes) over that time, and the card's name and power limit.
NeRFBlock: wall time of forward + backward (parameters, positions and directions) on `--block-points` points, ended by a
device synchronise, median of `--iters`.
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


def dinput_bytes(n: int) -> int:
    tiles = (n + 127) // 128
    return tiles * (4 + 4 + 2) * 128 * 128 + n * 3 * 4 * 4   # A panels + (positions, directions) read + two gradients written


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument('--samples', type=int, default=786_432)
    ap.add_argument('--iters', type=int, default=20)
    ap.add_argument('--block-points', type=int, default=1_000_000)
    args = ap.parse_args()
    from nerficg_b200 import ops, params
    from nerficg_b200.Methods.NeRF.Model import NeRFBlock
    torch.manual_seed(0)
    block = NeRFBlock(8, 1, 256, 10, 4, True, [5], 'relu').to(DEV)
    flat = block.flat_params
    res = {'card': card()}

    # ---- K4c alone ----
    n = args.samples
    pts = torch.rand(n, 3, device=DEV) * 4 - 2
    dirs = torch.nn.functional.normalize(torch.randn(n, 3, device=DEV), dim=-1)
    packed = ops.mlp_pack(flat)
    stash = torch.empty(ops.mlp_stash_bytes(n), dtype=torch.uint8, device=DEV)
    out = ops.mlp_forward(packed, flat, pts, torch.zeros_like(pts), dirs, torch.zeros(n, 1, device=DEV), None, stash)
    ws = torch.empty(ops.mlp_backward_workspace_bytes(n), dtype=torch.uint8, device=DEV)
    up = torch.randn(n, 4, device=DEV) * 10
    ops.mlp_backward_dgrad(up, out, stash, ws, packed, flat, n, 1)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=DEV)
    times = []
    for i in range(args.iters + 3):
        flush.fill_(i & 255)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        ops.mlp_backward_inputs(ws, flat, pts, dirs, n)
        b.record()
        b.synchronize()
        if i >= 3:
            times.append(a.elapsed_time(b) * 1e-3)
    t = sorted(times)[len(times) // 2]
    nbytes = dinput_bytes(n)
    res['k4c'] = {'samples': n, 'median_s': t, 'min_s': min(times), 'max_s': max(times), 'bytes': nbytes,
                  'bytes_per_s': nbytes / t, 'l2': 'overwritten before every launch'}
    del stash, ws, out, up, flush

    # ---- NeRFBlock forward + backward ----
    m = args.block_points
    pts = torch.rand(m, 3, device=DEV) * 4 - 2
    dirs = torch.nn.functional.normalize(torch.randn(m, 3, device=DEV), dim=-1)
    u_c, u_s = torch.randn(m, 3, device=DEV), torch.randn(m, 1, device=DEV)
    walls = []
    for i in range(args.iters + 2):
        block.zero_grad(set_to_none=True)
        p = pts.clone().requires_grad_(True)
        d = dirs.clone().requires_grad_(True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        sig, rgb = block(p, d)
        ((rgb * u_c).sum() + (sig * u_s).sum()).backward()
        torch.cuda.synchronize()
        if i >= 2:
            walls.append(time.perf_counter() - t0)
    res['block_fwd_bwd'] = {'points': m, 'median_s': sorted(walls)[len(walls) // 2], 'min_s': min(walls), 'max_s': max(walls),
                            'grads': 'parameters + positions + directions'}
    print(json.dumps(res))


if __name__ == '__main__':
    main()
