"""The C-ABI shared library loads and exports exactly what include/qsparse_b200.h declares
(no compute calls: there is no GPU in the CPU test tier)."""
import ctypes
import re
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent


def declared_symbols():
    text = (ROOT / "include" / "qsparse_b200.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(qsb_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_are_exported():
    from qsparse_b200.build import build
    lib_path = build()
    lib = ctypes.CDLL(str(lib_path))
    names = declared_symbols()
    assert len(names) >= 25
    for name in names:
        assert hasattr(lib, name), f"{name} declared in the header but not exported"


def test_python_binding_covers_header():
    from qsparse_b200 import _native
    assert sorted(_native.exported_symbols()) == declared_symbols()
    lib = _native.load_library()
    assert lib.qsb_abi_version() == 3
    assert b"bad argument" in lib.qsb_error_string(-1)


def test_argument_errors_without_gpu():
    """Argument validation happens before any CUDA call."""
    from qsparse_b200 import _native
    lib = _native.load_library()
    null = ctypes.c_void_p(0)
    assert lib.qsb_fq_pow2_fwd(null, null, null, 1, 5.0, null, 0, -1, 1, 1, null) == -1   # negative size
    assert lib.qsb_fq_pow2_fwd(null, null, null, 1, 5.0, null, 0, 0, 1, 1, null) == 0     # empty tensor: no-op
    assert lib.qsb_fq_pow2_fwd(null, null, null, 1, 5.0, null, 0, 1, 1, 8, null) == -1    # null pointers
    assert lib.qsb_kth_value(null, 0, 0, 0, null, null, 0, null) == -1
    assert lib.qsb_mask_apply(null, null, null, 0, 1, 1, 1, null) == -1                   # mask_kind none
    # the structured prune -> quantize parameter step on statistics rows: host buffers, never dereferenced
    c = 8
    mag, amax, scale, dec = ((ctypes.c_float * c)() for _ in range(4))
    mask, asum = (ctypes.c_uint8 * c)(), (ctypes.c_double * c)()

    def params(channels, n_rows=1, k=2, refresh=1):
        return lib.qsb_prune_quant_params(mag, mask, scale, dec, asum, amax, n_rows, 0, channels, 64.0, 1, 1,
                                          refresh, k, 8, 1, 1, null)
    assert params(0) == -4 and params(4097) == -4                                       # QSB_E_UNSUPPORTED
    assert params(c, n_rows=0) == -1
    assert params(c, k=c) == -1 and params(c, k=-1) == -1                               # k outside [0, C) on a refresh


def test_product_fails_loudly_on_cpu_tensors():
    import torch
    import qsparse_b200 as qs
    from qsparse_b200.quantize import quantize_with_decimal, quantize_with_line
    qs.set_qsparse_options(log_on_created=False)
    with pytest.raises(RuntimeError, match="CUDA-only"):
        quantize_with_decimal(torch.rand(8), 8, 5)
    with pytest.raises(RuntimeError, match="CUDA-only"):
        quantize_with_line(torch.rand(8))
    with pytest.raises(RuntimeError, match="CUDA-only"):
        qs.quantize(bits=8, timeout=1)(torch.rand(2, 4))
    with pytest.raises(RuntimeError, match="CUDA-only"):
        qs.prune(sparsity=0.5, start=0, interval=1)(torch.rand(2, 4))
    with pytest.raises(RuntimeError, match="CUDA-only"):
        qs.calculate_mask_given_importance(torch.rand(10), 0.5)


def test_product_never_imports_the_oracle():
    import subprocess
    import sys
    code = ("import sys; import qsparse_b200, qsparse_b200.fused, qsparse_b200.parallel, qsparse_b200.ops; "
            "bad=[m for m in sys.modules if m.split('.')[0]=='oracle']; assert not bad, bad")
    subprocess.run([sys.executable, "-c", code], check=True, cwd=str(ROOT))
    for py in (ROOT / "qsparse_b200").glob("*.py"):
        assert "oracle" not in py.read_text().replace("# oracle", ""), py
