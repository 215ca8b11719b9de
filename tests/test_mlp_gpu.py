"""K3/K4 parity: fused tcgen05 MLP against the oracle (fp32) with teacher-forced inputs."""
import pytest
import torch

from oracle import nerf_oracle as O

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


@pytest.fixture(scope='module')
def ops():
    from nerficg_b200 import ops
    return ops


@pytest.fixture(scope='module')
def net():
    from nerficg_b200 import ops, params
    sd = O.init_state_dict(0)
    flat = {p: params.flatten_state_dict(sd, p, DEV) for p in ('nerf.', 'coarse_nerf.')}
    packed = {p: ops.mlp_pack(f) for p, f in flat.items()}
    return sd, flat, packed


def test_points_golden(ops, net, golden):
    """NeRFBlock.forward on raw points (S = 1, origin = point, dir = 0): vs reference outputs."""
    sd, flat, packed = net
    g = golden('mlp')
    n = g['pts'].shape[0]
    zero = torch.zeros(n, 3, device=DEV)
    for prefix, ks, kc in (('nerf.', 'sigma', 'rgb'), ('coarse_nerf.', 'sigma_coarse', 'rgb_coarse')):
        out = ops.mlp_forward(packed[prefix], flat[prefix], g['pts'].to(DEV), zero, g['dirs'].to(DEV),
                              torch.zeros(n, 1, device=DEV)).cpu().reshape(n, 4)
        assert (out[:, :3] - g[kc]).abs().max() <= 1e-3
        assert (out[:, 3:] - g[ks]).abs().max() <= 1e-3 + 2e-3 * g[ks].abs().max()


@pytest.mark.parametrize('n_rays,s', [(1, 1), (3, 64), (100, 192), (37, 77), (1500, 64), (700, 192)])
def test_forward_vs_oracle(ops, net, n_rays, s):
    sd, flat, packed = net
    g = torch.Generator().manual_seed(n_rays + s)
    o = torch.randn(n_rays, 3, generator=g) * 2
    d = torch.randn(n_rays, 3, generator=g)
    vd = torch.nn.functional.normalize(d, dim=-1)
    z = torch.sort(2 + 4 * torch.rand(n_rays, s, generator=g), -1).values
    noise = torch.randn(n_rays * s, generator=g)
    x = o[:, None] + d[:, None] * z[..., None]
    sig, rgb = O.mlp_forward(sd, 'nerf.', x.reshape(-1, 3), vd[:, None].expand_as(x).reshape(-1, 3), noise[:, None])
    out = ops.mlp_forward(packed['nerf.'], flat['nerf.'], o.to(DEV), d.to(DEV), vd.to(DEV), z.to(DEV), noise.to(DEV))
    out = out.cpu().reshape(-1, 4)
    assert (out[:, :3] - rgb).abs().max() <= 1e-3, (out[:, :3] - rgb).abs().max()
    assert (out[:, 3:] - sig).abs().max() <= 1e-3 + 2e-3 * sig.abs().max(), (out[:, 3:] - sig).abs().max()
    # training variant (stash) must produce identical outputs
    stash = torch.empty(ops.mlp_stash_bytes(n_rays * s), dtype=torch.uint8, device=DEV)
    out_t = ops.mlp_forward(packed['nerf.'], flat['nerf.'], o.to(DEV), d.to(DEV), vd.to(DEV), z.to(DEV), noise.to(DEV), stash)
    assert torch.equal(out_t.cpu().reshape(-1, 4), out)


def _rel_l2(a, b, floor=0.0):
    return ((a - b).norm() / (b.norm() + floor + 1e-30)).item()


@pytest.mark.parametrize('n_rays,s,scale', [(64, 64, 1024.0), (300, 192, 4096.0), (5, 77, 2048.0), (2048, 64, 1024.0)])
def test_backward_vs_oracle(ops, net, n_rays, s, scale):
    """dL/dparams of NeRFBlock.forward for random upstream gradients.

    Stated tolerance (per-tensor relative L2): 2e-2 against the oracle evaluated with the same
    fp16 operand rounding as the tensor-core path, 1e-1 against the plain fp32 oracle -- the
    difference is ReLU units whose pre-activation lies within the fp16 forward error of zero and
    therefore switch on/off (each flip changes a gradient term by 100 %)."""
    from nerficg_b200 import params as P
    sd, flat, packed = net
    g = torch.Generator().manual_seed(7 * n_rays + s)
    o = torch.randn(n_rays, 3, generator=g) * 2
    d = torch.randn(n_rays, 3, generator=g)
    vd = torch.nn.functional.normalize(d, dim=-1)
    z = torch.sort(2 + 4 * torch.rand(n_rays, s, generator=g), -1).values
    up = torch.randn(n_rays * s, 4, generator=g) * 1e-3   # dL/d(r,g,b,sigma)
    x = o[:, None] + d[:, None] * z[..., None]
    ref = {}
    for tag, dt in (('fp32', None), ('fp16', torch.float16)):
        leaf = {k: v.clone().requires_grad_(True) for k, v in sd.items() if k.startswith('nerf.') and 'frequency' not in k}
        sig, rgb = O.mlp_forward({**sd, **leaf}, 'nerf.', x.reshape(-1, 3), vd[:, None].expand_as(x).reshape(-1, 3),
                                 operand_dtype=dt)
        ((rgb * up[:, :3]).sum() + (sig * up[:, 3:]).sum()).backward()
        ref[tag] = {k[len('nerf.'):]: v.grad for k, v in leaf.items()}
        sigma_on = (sig.detach() > 0).reshape(-1)      # density-ReLU mask of the fp16-operand oracle (last iteration)

    n = n_rays * s
    stash = torch.empty(ops.mlp_stash_bytes(n), dtype=torch.uint8, device=DEV)
    out = ops.mlp_forward(packed['nerf.'], flat['nerf.'], o.to(DEV), d.to(DEV), vd.to(DEV), z.to(DEV), None, stash)
    up_dev = up.to(DEV).clone()
    # K6 folds the density ReLU (relu_mask=1).  The oracle's mask is used so that a sample whose sigma_raw is
    # within rounding of zero cannot flip a whole term of the (tiny, cancellation-prone) density-bias gradient.
    assert ((out.reshape(-1, 4)[:, 3] > 0).cpu() != sigma_on).float().mean() <= 1e-2
    up_dev[:, 3] *= sigma_on.to(DEV)
    up_dev *= scale
    ws = torch.empty(ops.mlp_backward_workspace_bytes(n), dtype=torch.uint8, device=DEV)
    grads = torch.zeros_like(flat['nerf.'])
    ops.mlp_backward(grads, up_dev, out, stash, ws, packed['nerf.'], flat['nerf.'], n_rays, s, scale)
    torch.cuda.synchronize()
    got = P.views(grads.cpu())
    # the 1- and 3-element head biases are plain sums of the upstream gradients: with few samples they cancel to
    # nearly zero, so their error is measured against the size of the summands rather than of the (tiny) sum
    floor = {k: (0.05 * up.norm().item() if v.numel() <= 3 else 0.0) for k, v in got.items()}
    e16 = {k: round(_rel_l2(v, ref['fp16'][k], floor[k]), 4) for k, v in got.items()}
    e32 = {k: round(_rel_l2(v, ref['fp32'][k], floor[k]), 4) for k, v in got.items()}
    import json, os
    os.makedirs('gpurun_out', exist_ok=True)
    with open('gpurun_out/grad_parity.jsonl', 'a') as f:
        f.write(json.dumps({'n_rays': n_rays, 's': s, 'scale': scale, 'vs_fp16_oracle': e16, 'vs_fp32_oracle': e32}) + '\n')
    assert max(e16.values()) <= 2e-2, e16
    assert max(e32.values()) <= 1e-1, e32
    # accumulation semantics: a second call doubles the gradient
    ops.mlp_backward(grads, up_dev, out, stash, ws, packed['nerf.'], flat['nerf.'], n_rays, s, scale)
    got2 = P.views(grads.cpu())
    assert _rel_l2(got2['feature_layer.weight'], 2 * ref['fp16']['feature_layer.weight']) <= 2e-2
