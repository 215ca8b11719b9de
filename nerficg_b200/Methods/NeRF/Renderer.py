"""NeRF renderer: the reference's ``NeRFRayRenderingComponent`` / ``NeRFRenderer`` interface
(src/Methods/NeRF/Renderer.py) on top of the sm_100a kernels.

Per chunk of at most RAY_BATCH_SIZE rays (Renderer.py:45-47) the pipeline is
    K1 stratified depths -> K3 coarse MLP -> K5 composite (+weights) -> K2 inverse-CDF + merge
    -> K3 fine MLP -> K5 composite
with the same torch RNG draws in the same order as the reference (rand(n,Nc), [randn coarse noise],
rand(n,Nf), [randn fine noise]).  Differentiation goes through ONE autograd node per chunk whose backward runs, per
pass, K6 (compositing backward), then K4 (MLP dgrad + wgrad) when a parameter needs grad or K4a (dgrad only) when none
does, then K4r when a ray tensor needs grad: dL/d(origin, direction, view_direction) reduced per ray from the same
gradient stash (d also gets the compositing term, the interval lengths scale with |d|).  Without a ray tensor that
requires grad the backward is exactly the parameter-only one.
"""
from __future__ import annotations

import os

import torch

from ... import Framework, ops, params
from ...profiling import stage
from ...Cameras.Perspective import PerspectiveCamera
from ...Datasets.utils import RayBatch, View
from ...Logging import Logger
from ..Base.Model import BaseModel
from ..Base.Renderer import BaseRenderer, BaseRenderingComponent
from .Model import NeRF, NeRFBlock


def default_grad_scale(n_rays: int) -> float:
    """Static loss scale of the fp16 backward.  dL/drgb of an MSE over n rays is <= 2/(3n), so 16*n keeps the
    largest upstream value near 10 (fp16 max 65504) while lifting typical per-sample gradients (1e-8..1e-5
    unscaled) into the fp16 normal range.  Override with NERF_B200_GRAD_SCALE."""
    env = os.environ.get('NERF_B200_GRAD_SCALE')
    if env:
        return float(env)
    return float(min(max(16 * n_rays, 1024), 1 << 20))


class _Workspace:
    """Per-device scratch shared by all backward calls (they are serialised on one stream)."""
    buffers: dict = {}

    @classmethod
    def get(cls, device: torch.device, nbytes: int) -> torch.Tensor:
        buf = cls.buffers.get(device)
        if buf is None or buf.numel() < nbytes:
            buf = torch.empty(nbytes, dtype=torch.uint8, device=device)
            cls.buffers[device] = buf
        return buf


class _ChunkState:
    """Non-tensor arguments of one chunk (flat parameter buffers, weight images, constants)."""
    __slots__ = ('flat_c', 'flat_f', 'packed_c', 'packed_f', 'background', 'near', 'far', 'n_coarse', 'n_fine', 'need_grad')


class _RenderChunk(torch.autograd.Function):
    """rgb/depth/alpha (+coarse) of one ray chunk.  The trailing inputs are the model parameters (24 per block,
    flat-buffer order): they are only there so autograd routes the gradients, which are returned as views of one
    flat gradient buffer per block."""

    @staticmethod
    def forward(ctx, st: _ChunkState, origin, direction, view_direction, u_c, u_f, noise_c, noise_f, *model_params):
        n = origin.shape[0]
        dev = origin.device
        ctx.st = st
        ctx.set_materialize_grads(False)  # unused outputs (depth, alpha, coarse) arrive as None
        outs = []
        need = st.need_grad
        if st.n_coarse > 0:
            with stage('K1 stratified'):
                z_c = ops.sample_stratified(n, st.n_coarse, st.near, st.far, u_c, dev)
            stash_c = torch.empty(ops.mlp_stash_bytes(n * st.n_coarse), dtype=torch.uint8, device=dev) if need else None
            with stage('K3 mlp_fwd coarse'):
                rs_c = ops.mlp_forward(st.packed_c, st.flat_c, origin, direction, view_direction, z_c, noise_c, stash_c)
            with stage('K5 composite coarse'):
                rgb_c, depth_c, alpha_c, w_c = ops.composite_forward(z_c, rs_c, direction, st.background, want_weights=True)
            with stage('K2 importance+merge'):
                z = ops.sample_importance(z_c, w_c, st.n_fine, u_f)
            outs = [rgb_c, depth_c, alpha_c]
        else:
            with stage('K1 stratified'):
                z = ops.sample_stratified(n, st.n_fine, st.near, st.far, u_f, dev)
            z_c = rs_c = stash_c = None
        stash_f = torch.empty(ops.mlp_stash_bytes(z.numel()), dtype=torch.uint8, device=dev) if need else None
        with stage('K3 mlp_fwd fine'):
            rs_f = ops.mlp_forward(st.packed_f, st.flat_f, origin, direction, view_direction, z, noise_f, stash_f)
        with stage('K5 composite fine'):
            rgb, depth, alpha, _ = ops.composite_forward(z, rs_f, direction, st.background)
        if need:
            ctx.saved = (origin, direction, view_direction, z_c, rs_c, stash_c, z, rs_f, stash_f)
        return (rgb, depth, alpha, *outs)

    @staticmethod
    def backward(ctx, g_rgb, g_depth, g_alpha, g_rgb_c=None, g_depth_c=None, g_alpha_c=None):
        st = ctx.st
        n_blocks = 2 if st.n_coarse > 0 else 1
        if not st.need_grad:
            return (None,) * (8 + 24 * n_blocks)
        origin, direction, view_direction, z_c, rs_c, stash_c, z, rs_f, stash_f = ctx.saved
        n = z.shape[0]
        scale = default_grad_scale(n)
        ws = _Workspace.get(z.device, ops.mlp_backward_workspace_bytes(z.numel()))
        need_params = any(ctx.needs_input_grad[8:])
        # dL/d(origin, direction, view_direction): both passes add into these
        d_rays = [torch.zeros(n, 3, device=z.device) if need else None for need in ctx.needs_input_grad[1:4]]
        need_rays = any(t is not None for t in d_rays)

        def one(flat, packed, zz, rs, stash, gr, gd, ga):
            grad = torch.zeros_like(flat) if need_params else None
            if gr is None and gd is None and ga is None:
                return grad
            gr = torch.zeros(n, 3, device=zz.device) if gr is None else gr
            flatten = lambda t: None if t is None else t.reshape(-1)
            with stage('K6 composite_bwd'):
                d_rs = ops.composite_backward(zz, rs, direction, st.background, gr, flatten(gd), flatten(ga), True, scale)
            if need_params:
                with stage('K4 mlp_bwd (dgrad + wgrad)'):
                    ops.mlp_backward(grad, d_rs, rs, stash, ws, packed, flat, n, zz.shape[1], scale)
            else:
                with stage('K4a mlp_bwd dgrad'):
                    ops.mlp_backward_dgrad(d_rs, rs, stash, ws, packed, flat, n, zz.shape[1])
            if need_rays:  # before the next pass's dgrad overwrites ws
                with stage('K4r mlp_bwd rays'):
                    ops.mlp_backward_rays(*d_rays, ws, flat, origin, direction, view_direction, zz, rs, d_rs, scale)
            return grad

        def param_grads(grad):
            return [None] * 24 if grad is None else list(params.views(grad).values())

        grads = []
        if st.n_coarse > 0:
            grads += param_grads(one(st.flat_c, st.packed_c, z_c, rs_c, stash_c, g_rgb_c, g_depth_c, g_alpha_c))
        grads += param_grads(one(st.flat_f, st.packed_f, z, rs_f, stash_f, g_rgb, g_depth, g_alpha))
        ctx.saved = None
        return (None, *d_rays) + (None,) * 4 + tuple(grads)


class NeRFRayRenderingComponent(BaseRenderingComponent):
    def __init__(self, coarse_nerf: NeRFBlock | None, nerf: NeRFBlock) -> None:
        super().__init__()
        self.coarse_nerf = coarse_nerf
        self.nerf = nerf

    def forward(self, rays: RayBatch, camera: PerspectiveCamera, ray_batch_size: int, n_samples_coarse_nerf: int,
                n_samples_nerf: int, randomize_samples: bool, random_noise_density: float,
                noise: list[dict] | None = None) -> dict[str, torch.Tensor]:
        """Same contract as reference Renderer.py:29-95.  ``noise`` optionally supplies per-chunk dicts with
        ``u_c, u_f, n_c, n_f`` (uniform / already-scaled normal noise) instead of drawing from torch's RNG."""
        use_coarse = n_samples_coarse_nerf > 0
        if use_coarse and self.coarse_nerf is None:
            raise Framework.RendererError('coarse samples requested but the model has no coarse network')
        dev = rays.device
        st = _ChunkState()
        st.background = camera.background_color.to(device=dev, dtype=torch.float32).contiguous()
        st.near, st.far = float(camera.near_plane), float(camera.far_plane)
        st.n_coarse, st.n_fine = n_samples_coarse_nerf, n_samples_nerf
        blocks = ([self.coarse_nerf] if use_coarse else []) + [self.nerf]
        model_params = [p for b in blocks for p in b.ordered_parameters()]
        # stashes (and the backward weight images) are kept when a parameter or a ray tensor needs grad
        ray_tensors = (rays.origin, rays.direction, rays.view_direction)
        st.need_grad = torch.is_grad_enabled() and (any(p.requires_grad for p in model_params)
                                                    or any(t is not None and t.requires_grad for t in ray_tensors))
        st.flat_f = self.nerf.flat_params
        st.flat_c = self.coarse_nerf.flat_params if use_coarse else None
        # weight images are rebuilt on every call (15 us per block): parameters may have changed in place
        st.packed_f = ops.mlp_pack(st.flat_f, with_backward=st.need_grad)
        st.packed_c = ops.mlp_pack(st.flat_c, with_backward=st.need_grad) if use_coarse else None
        keys = ['rgb', 'depth', 'alpha'] + (['rgb_coarse', 'depth_coarse', 'alpha_coarse'] if use_coarse else [])
        outputs = {k: [] for k in keys}
        n_total = n_samples_coarse_nerf + n_samples_nerf
        for ci, chunk in enumerate(rays.split(ray_batch_size)):
            n = len(chunk)
            if chunk.view_direction is None:
                raise Framework.RendererError('NeRF needs RayBatch.view_direction')
            u_c = u_f = n_c = n_f = None
            if noise is not None:
                d = noise[ci]
                u_c, u_f, n_c, n_f = d.get('u_c'), d.get('u_f'), d.get('n_c'), d.get('n_f')
            else:
                # draw order of the reference (SURVEY 8b "Threading"): rand, [randn], rand, [randn]
                if use_coarse:
                    if randomize_samples:
                        u_c = torch.rand((n, n_samples_coarse_nerf), dtype=torch.float32, device=dev)
                    if random_noise_density > 0.0:
                        n_c = random_noise_density * torch.randn((n * n_samples_coarse_nerf, 1), dtype=torch.float32, device=dev)
                if randomize_samples:
                    u_f = torch.rand(n, n_samples_nerf, device=dev)
                if random_noise_density > 0.0:
                    n_f = random_noise_density * torch.randn((n * n_total, 1), dtype=torch.float32, device=dev)
            res = _RenderChunk.apply(st, chunk.origin.contiguous(), chunk.direction.contiguous(),
                                     chunk.view_direction.contiguous(), u_c, u_f, n_c, n_f, *model_params)
            for k, t in zip(keys, res):
                outputs[k].append(t)
        return {k: (torch.cat(v, dim=0) if len(v) > 1 else v[0]) for k, v in outputs.items()}


@Framework.Configurable.configure(
    RAY_BATCH_SIZE=8192,
    N_SAMPLES=256,
    COARSE_RATIO=0.25,
)
class NeRFRenderer(BaseRenderer):
    """Renderer of the NeRF method (reference Renderer.py:98-165)."""

    def __init__(self, model: BaseModel) -> None:
        super().__init__(model, [NeRF])
        if self.model.coarse_nerf is None:
            self.n_samples_coarse_nerf = 0
            self.n_samples_nerf = self.N_SAMPLES
            Logger.log_info(f'using {self.n_samples_nerf} samples per ray')
        else:
            self.n_samples_coarse_nerf = round(self.N_SAMPLES * self.COARSE_RATIO)
            self.n_samples_nerf = self.N_SAMPLES - self.n_samples_coarse_nerf
            Logger.log_info(f'using {self.n_samples_coarse_nerf} coarse and {self.n_samples_nerf} fine samples per ray')
        self.ray_rendering_component = NeRFRayRenderingComponent.get(self.model.coarse_nerf, self.model.nerf)

    def render_rays(self, rays: RayBatch, camera: PerspectiveCamera, randomize_samples: bool = False,
                    random_noise_density: float = 0.0, noise: list[dict] | None = None) -> dict[str, torch.Tensor]:
        return self.ray_rendering_component(rays, camera, self.RAY_BATCH_SIZE, self.n_samples_coarse_nerf,
                                            self.n_samples_nerf, randomize_samples, random_noise_density, noise)

    def render_image(self, view: View, to_chw: bool = False, benchmark: bool = False) -> dict[str, torch.Tensor]:
        with stage('K0 generate_rays'):
            rays = view.get_rays()
        rendered = self.render_rays(rays, view.camera)
        for key in rendered:
            rendered[key] = rendered[key].reshape(view.camera.height, view.camera.width, -1)
            if to_chw:
                rendered[key] = rendered[key].permute(2, 0, 1)
        return rendered

    def postprocess_outputs(self, outputs, view, dataset=None, index: int = 0) -> dict[str, torch.Tensor]:
        """3xHxW images in [0,1] (reference Renderer.py:142-165): clamped colour, alpha, and depth normalised to
        [near, far], coloured with the SPECTRAL map and masked by alpha."""
        from ...Visual import apply_color_map
        near_far = (view.camera.near_plane, view.camera.far_plane)
        out = {'rgb': outputs['rgb'].clamp_(0.0, 1.0), 'alpha': outputs['alpha'].expand_as(outputs['rgb']),
               'depth': apply_color_map('SPECTRAL', outputs['depth'], near_far, outputs['alpha'])}
        if self.n_samples_coarse_nerf > 0:
            out |= {'rgb_coarse': outputs['rgb_coarse'].clamp_(0.0, 1.0),
                    'alpha_coarse': outputs['alpha_coarse'].expand_as(outputs['rgb_coarse']),
                    'depth_coarse': apply_color_map('SPECTRAL', outputs['depth_coarse'], near_far, outputs['alpha_coarse'])}
        return out
