"""CPU: the C-ABI library loads and exports every symbol include/nerf_b200.h declares (no compute without a GPU)."""
import ctypes
import re
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
HEADER = ROOT / 'include' / 'nerf_b200.h'


def declared_symbols() -> list[str]:
    text = re.sub(r'/\*.*?\*/', '', HEADER.read_text(), flags=re.S)
    return sorted(set(re.findall(r'\b(nerf_[a-z0-9_]+)\s*\(', text)))


@pytest.fixture(scope='module')
def library():
    from nerficg_b200 import _lib
    if not _lib.LIB_PATH.exists():
        import __graft_entry__
        __graft_entry__.build()
    return _lib


def test_header_declares_the_stage_entry_points():
    names = declared_symbols()
    for stage in ('nerf_sample_stratified', 'nerf_sample_importance', 'nerf_mlp_forward', 'nerf_mlp_backward',
                  'nerf_composite_forward', 'nerf_composite_backward', 'nerf_mlp_pack', 'nerf_device_check', 'nerf_last_error'):
        assert stage in names


def test_library_exports_every_declared_symbol(library):
    lib = ctypes.CDLL(str(library.LIB_PATH))
    for name in declared_symbols():
        assert hasattr(lib, name), f'{name} is declared in nerf_b200.h but not exported'
    assert sorted(library.EXPORTED_SYMBOLS) == declared_symbols(), 'ctypes prototypes and header disagree'


def test_abi_version_and_layout_queries_work_without_gpu(library):
    lib = library.load()
    assert lib.nerf_abi_version() == 1
    off, size, total = library.param_layout()
    assert len(off) == 24 and total == 595848 and sum(size) == 595844      # 595,844 parameters per block (SURVEY A.6)
    assert all(o % 4 == 0 for o in off)
    assert lib.nerf_mlp_packed_bytes() >= 2 * 557696 * 2                   # forward + transposed (dgrad) fp16 images
    assert lib.nerf_mlp_stash_bytes(128) > 0
    assert lib.nerf_mlp_backward_workspace_bytes(128) == 638976             # one 128-sample tile of the gradient stash (624 KB)


def test_no_cpu_fallback(library):
    """Product ops must fail loudly on CPU tensors / without a B200 instead of computing elsewhere."""
    import torch
    from nerficg_b200 import ops
    with pytest.raises(library.NativeLibraryError):
        ops.composite_forward(torch.zeros(2, 4), torch.zeros(2, 4, 4), torch.ones(2, 3), None)
    with pytest.raises(library.NativeLibraryError):
        ops.sample_stratified(2, 4, 2.0, 6.0, None, torch.device('cpu'))
    if not torch.cuda.is_available():
        assert lib_rc(library) != 0


def lib_rc(library) -> int:
    return library.load().nerf_device_check(0)


def test_product_package_never_imports_the_oracle():
    for path in (ROOT / 'nerficg_b200').rglob('*.py'):
        text = path.read_text()
        assert not re.search(r'^\s*(from|import)\s+oracle\b', text, flags=re.M), f'{path} imports the oracle'


def test_new_entry_points_validate_arguments_without_gpu(library):
    """K0 / K8 argument checks return an error code and a message before any launch (no GPU needed)."""
    import ctypes
    lib = library.load()
    assert lib.nerf_loss_mse(None, None, None, None, None, None, None, None, None, None, None, None, 16, 1.0, 0.0, None) != 0
    assert b'loss_mse' in lib.nerf_last_error()
    c2w = (ctypes.c_double * 16)(*([1.0, 0, 0, 0, 0, 1.0, 0, 0, 0, 0, 1.0, 0, 0, 0, 0, 1.0]))
    assert lib.nerf_generate_rays(None, None, None, None, 100, c2w, 10, 10, 10.0, 10.0, 5.0, 5.0, None) != 0
    assert b'generate_rays' in lib.nerf_last_error()
    assert lib.nerf_generate_rays(None, None, None, None, 0, c2w, 10, 10, 10.0, 10.0, 5.0, 5.0, None) == 0   # empty batch is a no-op
    assert lib.nerf_gather_rays(None, None, None, None, None, None, None, None, None, None, None, 0, None) == 0
    assert lib.nerf_gather_rays(None, None, None, None, None, None, None, None, None, None, None, 8, None) != 0
