"""Builds development variants of the library (csrc/build.py tag=...) for A/B timing on the GPU box:

    python tools/variants.py            # builds every variant below into nerficg_b200/libnerf_b200.<tag>.so
    NERF_B200_LIB=nerficg_b200/libnerf_b200.<tag>.so python tools/kernel_timing.py
"""
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from nerficg_b200.csrc import build as B  # noqa: E402

VARIANTS = {
    'pipe': ('NERF_BWD_PIPE',),                  # nerf_mlp_backward runs the fused layer-stationary backward (mlp_bwd_pipe.cu)
}

if __name__ == '__main__':
    import importlib
    names = sys.argv[1:] or list(VARIANTS)
    for tag in names:
        importlib.reload(B)
        print(tag, B.build(defines=VARIANTS[tag], tag=tag))
