"""CPU-side checks of the native library: it builds, loads, and exports every symbol the header declares.
No kernel is launched here (no GPU in this container)."""
import ctypes
import os
import subprocess
import sys

import pytest

from sheeprl_b200 import lib as L


@pytest.fixture(scope="module")
def built():
    from sheeprl_b200.build import build

    return build()


def test_library_exports_every_declared_symbol(built):
    lib = ctypes.CDLL(built)
    names = L.declared_symbols()
    assert len(names) >= 40
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, missing


def test_library_identity(built):
    lib = L.load_library()
    assert lib.b200rl_abi_version() == 1
    assert lib.b200rl_build_arch() == b"sm_100a"


def test_product_path_refuses_to_run_without_gpu():
    # in a process that sees no device, so that the check also runs on a machine with a GPU
    code = ("import pytest\n"
            "from sheeprl_b200 import lib as L\n"
            "from sheeprl_b200.configs import make_dv3_cfg\n"
            "from sheeprl_b200.engine import DV3Engine\n"
            "with pytest.raises(L.B200RLError):\n"
            "    DV3Engine(make_dv3_cfg('S', per_rank_batch_size=2, per_rank_sequence_length=2), (2,), device='cuda')\n")
    root = os.path.dirname(os.path.dirname(os.path.abspath(L.__file__)))
    r = subprocess.run([sys.executable, "-c", code], cwd=root, capture_output=True, text=True,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 0, r.stderr[-2000:]


def test_product_never_imports_oracle():
    root = os.path.dirname(os.path.abspath(L.__file__))
    for dp, _, files in os.walk(root):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dp, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, os.path.join(dp, f)
