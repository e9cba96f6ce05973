"""CPU: the C-ABI library builds/loads and exports every symbol include/kpf_b200.h declares (no compute calls)."""
import ctypes
import os

import pytest

from keypointfusion_b200 import _lib


def test_header_declares_entry_points():
    protos = _lib.parse_header()
    assert "kpf_getpcl" in protos and "kpf_img2pcl_index" in protos and "kpf_cross_decoder_layer" in protos
    assert all(params[-1][1] == "stream" for name, params in protos.items() if name != "kpf_abi_version")


def test_library_exports_every_declared_symbol():
    from keypointfusion_b200 import build
    if os.path.exists(build.NVCC):
        build.build()  # incremental: recompiles only stale objects
    L = ctypes.CDLL(_lib.LIB_PATH)
    for name in _lib.parse_header():
        assert hasattr(L, name), f"{name} declared in kpf_b200.h but not exported"
    assert _lib.lib().kpf_abi_version() >= 1


def test_split_selftest_refuses_unsupported_k():
    """The split-precision self-test has kernels for K in {16, 32, 64, 128, 256} only: any other K is refused before a launch,
    never run as a 256-deep GEMM over whatever memory follows the operands."""
    L = _lib.lib()
    for K in (48, 80, 240, 512):
        assert L.kpf_umma_split_selftest(None, None, None, 128, K, 0, 0, 0, None, None) == -1   # KPF_ERR_BAD_ARGUMENT


def test_no_fallback_on_cpu_tensors():
    import torch
    from keypointfusion_b200 import ops
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.uvd2xyz(torch.zeros(1, 2, 3), torch.zeros(1, 3), torch.eye(3)[None], torch.ones(1, 3), torch.ones(1, 4), 128)


def test_product_never_touches_the_oracle():
    """The oracle is test infrastructure: no module of the package (nor the C sources) may import, link or execute it."""
    import ast
    import glob
    import os
    root = os.path.join(os.path.dirname(__file__), "..", "keypointfusion_b200")
    for path in glob.glob(os.path.join(root, "**", "*.py"), recursive=True):
        tree = ast.parse(open(path).read())
        for node in ast.walk(tree):
            names = []
            if isinstance(node, ast.Import):
                names = [a.name for a in node.names]
            elif isinstance(node, ast.ImportFrom):
                names = [node.module or ""]
            assert not any(n.split(".")[0] == "oracle" for n in names), f"{path} imports the oracle"
    for path in glob.glob(os.path.join(root, "csrc", "*")):
        assert "oracle/" not in open(path, errors="ignore").read().replace("oracle/kpf_oracle.py", ""), path


def test_kernels_read_no_environment():
    """A kernel's code path is chosen by its arguments and inputs alone, never by an environment variable read inside the library."""
    import glob
    import os
    import re
    root = os.path.join(os.path.dirname(__file__), "..", "keypointfusion_b200", "csrc")
    srcs = glob.glob(os.path.join(root, "*"))
    assert srcs
    for path in srcs:
        assert not re.search(r"\bgetenv\s*\(", open(path, errors="ignore").read()), f"{path} calls getenv"
