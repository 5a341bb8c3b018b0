"""CPU tier: the C-ABI library builds for sm_100a, loads without a GPU driver, exports every
symbol include/triad_b200.h declares, and validates arguments before touching CUDA."""
import ctypes
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "triad_b200.h")


@pytest.fixture(scope="module")
def lib():
    from triad_b200 import build, _lib
    build.build()
    return _lib.load()


def declared_symbols():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(triad_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_are_exported(lib):
    from triad_b200 import _lib
    names = declared_symbols()
    assert len(names) >= 15
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/triad_b200.h but not exported"
        assert n in _lib.SIGNATURES, f"{n} has no ctypes signature in triad_b200/_lib.py"
    assert set(_lib.SIGNATURES) == set(names)


def test_library_is_self_contained():
    from triad_b200 import _lib
    out = subprocess.run(["ldd", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "libcuda.so" not in out and "libtorch" not in out and "not found" not in out


def test_sass_is_blackwell_native():
    """tcgen05.mma -> UTCHMMA, tcgen05.ld -> LDTM, TMA -> UTMALDG (B200_PROFILING.md)."""
    from triad_b200 import _lib
    r = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True)
    if r.returncode != 0:
        pytest.skip("cuobjdump unavailable")
    for mnemonic in ("UTCHMMA", "LDTM", "UTMALDG"):
        assert mnemonic in r.stdout, mnemonic
    assert "HGMMA" not in r.stdout


def test_status_strings_and_version(lib):
    assert lib.triad_abi_version() == 1
    assert lib.triad_status_string(0) == b"ok"
    for s in range(-8, 0):
        assert lib.triad_status_string(s) not in (b"", b"unknown status")


def test_argument_validation_without_gpu(lib):
    """Every entry point rejects bad arguments before any CUDA call (so this runs on CPU)."""
    E = {"arg": -1, "shape": -2, "align": -3, "ws": -4, "unsupported": -7}
    null = None
    one = ctypes.c_void_p(16)     # a non-null, 16-byte aligned fake pointer: never dereferenced on these paths
    odd = ctypes.c_void_p(24)
    assert lib.triad_row_scale(null, 4, 4, null, null) == E["arg"]
    assert lib.triad_row_scale(null, 0, 4, one, null) == E["shape"]
    f = lib.triad_maxmean_fwd
    assert f(null, one, one, one, 2, 2, 4, 8, 64, 1, one, null, one, 1 << 20, 0, null) == E["arg"]
    assert f(one, one, one, one, 2, 2, 4, 8, 60, 1, one, null, one, 1 << 20, 0, null) == E["shape"]   # D % 8
    assert f(one, one, one, one, 2, 2, 4, 8, 64, 7, one, null, one, 1 << 20, 0, null) == E["arg"]     # dtype
    assert f(odd, one, one, one, 2, 2, 4, 8, 64, 1, one, null, one, 1 << 20, 0, null) == E["align"]
    assert f(one, one, one, one, 2, 2, 4, 8, 64, 1, one, null, one, 16, 0, null) == E["ws"]
    assert lib.triad_last_error() != b""
    assert lib.triad_maxmean_fwd_workspace_bytes(2, 2, 4, 8, 64, 1) >= 256
    assert lib.triad_infonce_partial(null, 4, 4, 0, one, one, one, 1 << 20, null) == E["arg"]
    assert lib.triad_infonce_partial(one, 4, 4, 2, one, one, one, 1 << 20, null) == E["shape"]        # row0+rows > B
    assert lib.triad_infonce_finish(one, 4, 4, 0, one, one, 1, 1.0, one, one, one, 8, null) == E["ws"]
    b = lib.triad_maxmean_bwd
    assert b(one, one, null, one, one, one, one, 2, 2, 4, 8, 64, 1, one, one, 0, one, one, 256, 0, null) == E["arg"]
    assert b(one, one, one, one, one, one, one, 2, 2, 4, 8, 63, 1, one, one, 0, one, one, 256, 0, null) == E["shape"]
    # a flag bit the library does not define is rejected, not ignored (these reach the workspace check otherwise)
    assert b(one, one, one, one, one, one, one, 2, 2, 4, 8, 64, 1, one, one, 0, one, one, 256, 32, null) == E["ws"]
    for bad in (4, 8, 64, 512, 32 | 64):
        assert b(one, one, one, one, one, one, one, 2, 2, 4, 8, 64, 1, one, one, 0, one, one, 256, bad, null) == E["arg"], bad
    # dv beyond the largest patch count the dv sorts handle: rejected before any work is queued
    for dtype in (0, 1):
        ws = lib.triad_maxmean_bwd_workspace_bytes(2, 2, 4, 3073, 64, dtype)
        assert b(one, one, one, one, one, one, one, 2, 2, 4, 3073, 64, dtype, one, one, 0, one, one, ws, 0, null) == E["unsupported"], dtype
    assert lib.triad_topk(one, 10, 11, one, one, one, 1 << 20, null) == E["shape"]
    assert lib.triad_diag_ranks(null, 4, one, null) == E["arg"]
    assert lib.triad_similarity_matrix(one, one, one, 0, 1, 1, 8, one, null) == E["shape"]
    assert lib.triad_retrieve_scores(one, 4, one, 3, 8, 64, 1, one, 1, 2, one, one, 1 << 30, null) == E["arg"]   # direction
    n = lib.triad_nonneg_chunk
    assert n(null, 8, 1, one, -60.0, 1e-3, 1, one, one, 1 << 20, null) == E["arg"]
    assert n(one, 0, 1, one, -60.0, 1e-3, 1, one, one, 1 << 20, null) == E["shape"]
    assert n(one, 8, 1, one, 1.0, 1e-3, 1, one, one, 1 << 20, null) == E["arg"]           # lo must be negative
    assert n(odd, 8, 1, one, -60.0, 1e-3, 1, one, one, 1 << 20, null) == E["align"]
    assert n(one, 8, 1, one, -60.0, 1e-3, 1, one, one, 8, null) == E["ws"]
    assert lib.triad_nonneg_workspace_bytes() > 0
    # the packed (masked-query) forward needs room for the packed copy of q and the row maps
    base = lib.triad_maxmean_fwd_workspace_bytes_ex(4, 4, 8, 16, 64, 1, 0)
    assert base == lib.triad_maxmean_fwd_workspace_bytes(4, 4, 8, 16, 64, 1)
    assert lib.triad_maxmean_fwd_workspace_bytes_ex(4, 4, 8, 16, 64, 1, 16) >= 4 * 8 * 64 * 2 + 256
    assert lib.triad_maxmean_fwd_workspace_bytes_ex(4, 4, 8, 16, 64, 0, 16) == base      # fp32: never packed
    assert f(one, one, one, one, 2, 2, 4, 8, 64, 1, one, null, one, base, 16, null) == E["ws"]   # PACK_ROWS needs more
    assert isinstance(lib.triad_launch_count(), int)


def test_product_has_no_oracle_or_cpu_fallback():
    """The package must never import the oracle, and must fail loudly off-GPU."""
    import torch
    import triad_b200
    for root, _, files in os.walk(os.path.join(ROOT, "triad_b200")):
        for fn in files:
            if fn.endswith(".py"):
                src = open(os.path.join(root, fn)).read()
                assert "import oracle" not in src and "from oracle" not in src, fn
    m = triad_b200.TriadHotPath()
    a, v = torch.randn(2, 3, 64), torch.randn(2, 5, 64)
    with pytest.raises(RuntimeError):
        m.compute_all_similarities_av(a, v)
