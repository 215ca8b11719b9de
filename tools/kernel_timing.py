"""In-kernel stall accounting of the MLP kernels (nerf_debug_set_timing): where the MMA issuer, the weight producer
and one epilogue thread of every CTA spend their cycles.  Development aid; prints averages per CTA in cycles."""
import os
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from nerficg_b200 import _lib, ops, params  # noqa: E402

if os.environ.get('NERF_B200_LIB'):  # development: time another build of the library
    _lib.LIB_PATH = Path(os.environ['NERF_B200_LIB']).resolve()

DEV = 'cuda:0'
NAMES = ['mma wait A-ready', 'mma wait W-full', 'mma total', 'producer wait W-empty', 'producer total',
         'epilogue wait ACC-ready', 'epilogue total', 'epilogue stash drain', 'epilogue prologue', 'ctas']


def report(buf, base, title, ms):
    v = buf[base:base + 10].tolist()
    n = max(v[9], 1)
    print(f'--- {title}: {ms:.3f} ms')
    for name, x in zip(NAMES[:9], v[:9]):
        print(f'    {name:26s} {x / n:12.0f} cyc/CTA')
    if base == 0:   # forward only: waits of one epilogue thread that the table above counts as busy time
        for name, x in zip(('epilogue wait bias', 'epilogue slot barrier', 'epilogue mask store'), buf[22:25].tolist()):
            print(f'    {name:26s} {x / n:12.0f} cyc/CTA')


def main():
    args = [a for a in sys.argv[1:] if not a.startswith('--')]
    n_rays, s = (int(args[0]), int(args[1])) if len(args) > 1 else (4096, 192)
    g = torch.Generator().manual_seed(0)
    flat = (torch.rand(params.layout()[2], generator=g) - 0.5).mul(0.12).to(DEV)
    packed = ops.mlp_pack(flat)
    o = torch.randn(n_rays, 3, generator=g).to(DEV) * 0.1
    d = torch.nn.functional.normalize(torch.randn(n_rays, 3, generator=g), dim=-1).to(DEV)
    z = torch.sort(2 + 4 * torch.rand(n_rays, s, generator=g), -1).values.to(DEV)
    n = n_rays * s
    stash = torch.empty(ops.mlp_stash_bytes(n), dtype=torch.uint8, device=DEV)
    ws = torch.empty(ops.mlp_backward_workspace_bytes(n), dtype=torch.uint8, device=DEV)
    grads = torch.zeros_like(flat)
    up = torch.randn(n, 4, device=DEV) * 1e-3 * 1024
    buf = torch.zeros(64, dtype=torch.int64, device=DEV)

    noprof = '--noprof' in sys.argv   # time the PRODUCTION instantiations (the stall counters live in their own ones)

    def timed(fn):
        for _ in range(2):
            fn()
        buf.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if noprof:
            best = 1e9
            for _ in range(5):
                a.record()
                out = fn()
                b.record()
                torch.cuda.synchronize()
                best = min(best, a.elapsed_time(b))
            return out, best
        _lib.load().nerf_debug_set_timing(buf.data_ptr())
        a.record()
        out = fn()
        b.record()
        torch.cuda.synchronize()
        _lib.load().nerf_debug_set_timing(None)
        return out, a.elapsed_time(b)

    _, ms = timed(lambda: ops.mlp_forward(packed, flat, o, d, d, z))
    report(buf, 0, f'forward (inference) {n_rays}x{s}', ms)
    out, ms = timed(lambda: ops.mlp_forward(packed, flat, o, d, d, z, None, stash))
    report(buf, 0, f'forward (training)  {n_rays}x{s}', ms)
    _, ms = timed(lambda: ops.mlp_backward_dgrad(up, out, stash, ws, packed, flat, n_rays, s))
    report(buf, 10, f'dgrad               {n_rays}x{s}', ms)
    v = buf[20:22].tolist()
    n_cta = max(buf[19].item(), 1)
    print(f'    prologue: loads+arithmetic {v[0] / n_cta:12.0f} cyc/CTA, store drain {v[1] / n_cta:12.0f} cyc/CTA')
    print(f'    epilogue wait mask words   {buf[25].item() / n_cta:12.0f} cyc/CTA')
    for _ in range(3):
        ops.mlp_backward_wgrad(grads, stash, ws, n_rays, s, 1024.0)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    ops.mlp_backward_wgrad(grads, stash, ws, n_rays, s, 1024.0)
    b.record()
    torch.cuda.synchronize()
    print(f'--- wgrad {n_rays}x{s}: {a.elapsed_time(b):.3f} ms')


if __name__ == '__main__':
    main()
