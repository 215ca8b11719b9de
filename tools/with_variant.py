"""Runs pytest or a script of this repository against another build of the library, e.g. one built from an older checkout
for an A/B comparison:

    python tools/with_variant.py path/to/libnerf_b200.so pytest tests/test_mlp_gpu.py -m gpu -q
    python tools/with_variant.py path/to/libnerf_b200.so bench.py --steps 30 --warmup 5

The product binding (nerficg_b200/_lib.py) has no override of its own: this wrapper repoints it before anything loads it.
"""
import runpy
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from nerficg_b200 import _lib  # noqa: E402

if __name__ == '__main__':
    lib, target, *args = sys.argv[1:]
    _lib.LIB_PATH = Path(lib).resolve()
    assert _lib.LIB_PATH.exists(), _lib.LIB_PATH
    if target == 'pytest':
        import pytest
        raise SystemExit(pytest.main(args))
    sys.argv = [target] + args
    runpy.run_path(str(ROOT / target), run_name='__main__')
