"""The C-ABI library builds, loads, and exports every symbol include/nvf_b200.h declares
(no compute calls: there is no GPU in the CPU test tier)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_functions():
    src = open(os.path.join(ROOT, "include", "nvf_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(nvf_[a-z0-9_]+)\s*\(", src)))


def test_header_declares_expected_entry_points():
    names = declared_functions()
    for n in ("nvf_decode", "nvf_emit_points", "nvf_train_forward", "nvf_loss_seeds", "nvf_train_backward",
              "nvf_workspace_bytes", "nvf_strerror"):
        assert n in names


def test_cuda_library_builds_and_exports_all_symbols():
    from nvfpcc_b200 import build
    path = build.build()
    lib = ctypes.CDLL(path)
    for n in declared_functions():
        assert hasattr(lib, n), n
    lib.nvf_strerror.restype = ctypes.c_char_p
    assert lib.nvf_abi_version() == 1
    assert lib.nvf_strerror(-2) == b"unsupported channel configuration"


def test_binding_signature_table_matches_header():
    from nvfpcc_b200 import _lib
    assert sorted(_lib.EXPORTS) == declared_functions()


def test_workspace_query_needs_no_device():
    from nvfpcc_b200 import _lib, build
    b = _lib.Binding(build.build())
    d = b.desc(3, (8, 16, 8, 8))
    assert b.workspace_bytes(d, 1247, _lib.NVF_MODE_DECODE) > 1247 * 4096
    assert b.workspace_bytes(d, 16, _lib.NVF_MODE_TRAIN) > 16 * 2 * 2_700_000
    bad = b.desc(3, (8, 16, 8, 7))
    with pytest.raises(_lib.NvfError):
        b.workspace_bytes(bad, 1, _lib.NVF_MODE_DECODE)


def test_product_path_has_no_cpu_fallback():
    """Calling the product ops without a GPU must fail loudly, never fall back."""
    from tests.helpers import run_without_gpu
    run_without_gpu("import pytest, torch\n"
                    "from nvfpcc_b200 import ops\n"
                    "assert not torch.cuda.is_available()\n"
                    "with pytest.raises(RuntimeError):\n"
                    "    ops.decode_blocks(3, (8, 16, 8, 8), {}, torch.zeros(1, 3, 2, 2, 2), None, 0.5)\n")
