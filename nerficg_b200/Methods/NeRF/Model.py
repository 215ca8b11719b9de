"""NeRF model with the reference's module tree and state-dict keys (src/Methods/NeRF/Model.py), whose
parameters live in ONE flat fp32 buffer per block so the CUDA kernels, Adam and NCCL each see a single pointer."""
from __future__ import annotations

import torch
from torch.autograd.function import once_differentiable

from ... import Framework, ops, params
from ..Base.Model import BaseModel
from .utils import SUPPORTED_ACTIVATIONS, FrequencyEncoding


class NeRFBlock(torch.nn.Module):
    """position, direction -> density, colour.  Same constructor, submodule names and parameter shapes as the
    reference block (Model.py:13-57).  The CUDA path is specialised for the shipped architecture; any other
    combination raises (there is no fallback)."""

    def __init__(self, n_layers: int, n_color_layers: int, n_features: int, n_frequencies_position: int,
                 n_frequencies_direction: int, encoding_append_input: bool, input_skips: list[int],
                 activation_function: str) -> None:
        super().__init__()
        if activation_function not in SUPPORTED_ACTIVATIONS:
            raise Framework.ModelError(f'Invalid activation function "{activation_function}" (CUDA path supports {SUPPORTED_ACTIVATIONS})')
        arch = (n_layers, n_color_layers, n_features, n_frequencies_position, n_frequencies_direction,
                bool(encoding_append_input), list(input_skips))
        if arch != (8, 1, 256, 10, 4, True, [5]):
            raise Framework.ModelError(
                f'the sm_100a NeRF kernels are specialised for N_LAYERS=8, N_COLOR_LAYERS=1, N_FEATURES=256, '
                f'N_FREQUENCIES_POSITION=10, N_FREQUENCIES_DIRECTION=4, ENCODING_APPEND_INPUT=True, INPUT_SKIPS=[5]; got {arch}')
        self.input_skips = input_skips
        self.encoding_position = FrequencyEncoding(n_frequencies_position, encoding_append_input)
        self.encoding_direction = FrequencyEncoding(n_frequencies_direction, encoding_append_input)
        n_pos = self.encoding_position.get_n_outputs(3)
        n_dir = self.encoding_direction.get_n_outputs(3)
        relu = lambda: torch.nn.ReLU(True)
        # constructed in the reference's order so the same seed yields the same initial weights
        layers = [torch.nn.Sequential(torch.nn.Linear(n_pos, n_features, bias=True), relu())]
        for i in range(1, n_layers):
            layers.append(torch.nn.Sequential(
                torch.nn.Linear(n_features + (n_pos if i in input_skips else 0), n_features, bias=True), relu()))
        self.initial_layers = torch.nn.ModuleList(layers)
        self.feature_layer = torch.nn.Linear(n_features, n_features, bias=True)
        self.density_layer = torch.nn.Linear(n_features, 1, bias=True)
        self.density_activation = relu()
        self.color_layers = torch.nn.Sequential(torch.nn.Linear(n_features + n_dir, n_features // 2, bias=True), relu(),
                                                torch.nn.Linear(n_features // 2, 3, bias=True), torch.nn.Sigmoid())
        self._flat: torch.Tensor | None = None
        self._alias()

    # ---- flat storage ----------------------------------------------------------------------
    def _named(self) -> dict[str, torch.nn.Parameter]:
        named = dict(self.named_parameters())
        return {name: named[name] for name, _ in params.TENSOR_SPECS}

    def ordered_parameters(self) -> list[torch.nn.Parameter]:
        """The 24 parameters in flat-buffer order."""
        return list(self._named().values())

    def _alias(self) -> None:
        """(Re)creates the flat buffer on the parameters' device and makes every parameter a view into it."""
        named = self._named()
        device = next(iter(named.values())).device
        flat = torch.zeros(params.layout()[2], dtype=torch.float32, device=device)
        with torch.no_grad():
            for name, view in params.views(flat).items():
                view.copy_(named[name].data)
                named[name].data = view
        self._flat = flat

    def _apply(self, fn, recurse=True):
        super()._apply(fn, recurse)
        self._alias()
        return self

    @property
    def flat_params(self) -> torch.Tensor:
        """The block's parameters as one contiguous fp32 tensor (padding elements are zero)."""
        named = self._named()
        first = named[params.TENSOR_SPECS[0][0]]
        if self._flat is None or first.data_ptr() != self._flat.data_ptr():
            self._alias()
        return self._flat

    def forward(self, positions: torch.Tensor, directions: torch.Tensor, random_noise_density: float = 0.0):
        """The reference signature (Model.py:59-83): (N,3),(N,3) -> density (N,1), colour (N,3).

        Differentiable with respect to the 24 parameters, the positions and the directions whenever grad is enabled
        and any of them requires grad.  That pass keeps the activation stash for the backward: 676 KB per 128 points
        (plus 624 KB per 128 points of gradient workspace during the backward).  Otherwise the outputs carry no
        ``grad_fn`` and nothing is stashed."""
        flat = self.flat_params
        n = positions.shape[0]
        noise = random_noise_density * torch.randn(n, device=positions.device) if random_noise_density > 0.0 else None
        model_params = self.ordered_parameters()
        if torch.is_grad_enabled() and (positions.requires_grad or directions.requires_grad
                                        or any(p.requires_grad for p in model_params)):
            return _BlockFunction.apply(flat, noise, positions, directions, *model_params)
        with torch.no_grad():
            packed = ops.mlp_pack(flat, with_backward=False)
            out = ops.mlp_forward(packed, flat, positions, torch.zeros_like(positions), directions,
                                  torch.zeros(n, 1, device=positions.device), noise).reshape(n, 4)
        return out[:, 3:], out[:, :3]


class _BlockFunction(torch.autograd.Function):
    """NeRFBlock.forward with a backward: K3 with stash forward; K4 (dgrad, and wgrad when a parameter needs grad) and
    K4c (input gradients) backward.  Parameter gradients are returned as views of one flat gradient buffer."""

    @staticmethod
    def forward(ctx, flat, noise, positions, directions, *model_params):
        n = positions.shape[0]
        dev = positions.device
        ctx.set_materialize_grads(False)
        packed = ops.mlp_pack(flat, with_backward=True)
        stash = torch.empty(ops.mlp_stash_bytes(n), dtype=torch.uint8, device=dev)
        out = ops.mlp_forward(packed, flat, positions, torch.zeros_like(positions), directions, torch.zeros(n, 1, device=dev),
                              noise, stash).reshape(n, 4)
        ctx.save_for_backward(positions, directions)
        ctx.state = (flat, packed, stash, out)
        return out[:, 3:].clone(), out[:, :3].clone()

    @staticmethod
    @once_differentiable
    def backward(ctx, g_sigma, g_rgb):
        from .Renderer import _Workspace  # (Renderer imports this module)
        positions, directions = ctx.saved_tensors
        flat, packed, stash, out = ctx.state
        ctx.state = None
        need_pos, need_dir = ctx.needs_input_grad[2], ctx.needs_input_grad[3]
        need_params = ctx.needs_input_grad[4:]
        n = positions.shape[0]
        none = (None,) * 4 + (None,) * len(need_params)
        if n == 0 or (g_sigma is None and g_rgb is None):
            return none
        d_rs = torch.zeros(n, 4, dtype=torch.float32, device=positions.device)
        if g_rgb is not None:
            d_rs[:, :3] = g_rgb
        if g_sigma is not None:
            d_rs[:, 3] = g_sigma.reshape(n) * (out[:, 3] > 0)      # density ReLU, ReLU'(0) = 0
        # Loss scale of the fp16 gradient stash, from the upstream gradient itself and without a host synchronisation:
        # the power of two 2^k that brings max|d_rs| into [8, 16), the headroom the renderer's static scale aims at.
        _, e = torch.frexp(d_rs.abs().amax())
        k = (4 - e).clamp(-126, 126).float()
        d_rs *= torch.exp2(k)
        ws = _Workspace.get(positions.device, ops.mlp_backward_workspace_bytes(n))
        grad = None
        if any(need_params):
            grad = torch.zeros_like(flat)
            ops.mlp_backward(grad, d_rs, out, stash, ws, packed, flat, n, 1, 1.0)
            grad *= torch.exp2(-k)
        else:
            ops.mlp_backward_dgrad(d_rs, out, stash, ws, packed, flat, n, 1)
        d_pos = d_dir = None
        if need_pos or need_dir:
            d_pos, d_dir = ops.mlp_backward_inputs(ws, flat, positions if need_pos else None,
                                                   directions if need_dir else None, n)
            for t in (d_pos, d_dir):
                if t is not None:
                    t *= torch.exp2(-k)
        param_grads = [None] * len(need_params) if grad is None else \
            [v if need else None for v, need in zip(params.views(grad).values(), need_params)]
        return (None, None, d_pos, d_dir, *param_grads)


@Framework.Configurable.configure(
    HIERARCHICAL=True,
    N_LAYERS=8,
    N_COLOR_LAYERS=1,
    N_FEATURES=256,
    N_FREQUENCIES_POSITION=10,
    N_FREQUENCIES_DIRECTION=4,
    ENCODING_APPEND_INPUT=True,
    INPUT_SKIPS=[5],
    NETWORK_ACTIVATION='relu',
)
class NeRF(BaseModel):
    """Coarse + fine NeRFBlock (Model.py:86-128)."""

    def __init__(self, name: str = None) -> None:
        super().__init__(name)
        self.coarse_nerf: NeRFBlock | None = None
        self.nerf: NeRFBlock | None = None

    def _block(self) -> NeRFBlock:
        return NeRFBlock(self.N_LAYERS, self.N_COLOR_LAYERS, self.N_FEATURES, self.N_FREQUENCIES_POSITION,
                         self.N_FREQUENCIES_DIRECTION, self.ENCODING_APPEND_INPUT, self.INPUT_SKIPS, self.NETWORK_ACTIVATION)

    def build(self) -> 'NeRF':
        if self.HIERARCHICAL:
            self.coarse_nerf = self._block()
        self.nerf = self._block()
        return self

    def blocks(self) -> list[NeRFBlock]:
        return [b for b in (self.coarse_nerf, self.nerf) if b is not None]
