"""CPU tier of the e4m3 ragged caption gallery: the argument checks of triad_ragged_pack_e4m3 and
triad_retrieve_scores_ragged_e4m3, which must reject bad arguments before any CUDA call, and the Python-side
validation of RaggedGallery's fp8 storage."""
import ctypes

import numpy as np
import pytest
import torch

from triad_b200 import _lib, build
from triad_b200.retrieval import RaggedGallery, ragged_plan

SLOT = 256


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _lib.load()


def test_pack_e4m3_rejects_bad_arguments(lib):
    buf = ctypes.create_string_buffer(4096)
    p16 = (ctypes.addressof(buf) + 15) // 16 * 16

    def call(src=p16, dtype=1, src_rows=4, D=128, rowmap=p16, dst_rows=256, codes=p16, scales=p16):
        return lib.triad_ragged_pack_e4m3(src, dtype, src_rows, D, rowmap, dst_rows, codes, scales, None)

    for name in ("src", "rowmap", "codes", "scales"):
        assert call(**{name: None}) == -1, name                                   # TRIAD_ERR_BAD_ARG
    assert call(dtype=7) == -1
    assert call(src_rows=0) == -2 and call(dst_rows=100) == -2 and call(dst_rows=0) == -2   # TRIAD_ERR_BAD_SHAPE
    assert call(src_rows=1 << 31) == -2 and call(dst_rows=SLOT << 23) == -2
    for D in (0, 64, 192, 640):
        assert call(D=D) == -7, D                                                 # TRIAD_ERR_UNSUPPORTED
    assert call(src=p16 + 8) == -3 and call(codes=p16 + 8) == -3                  # TRIAD_ERR_ALIGNMENT
    assert call(rowmap=p16 + 2) == -3 and call(scales=p16 + 2) == -3


def test_scores_ragged_e4m3_rejects_bad_arguments(lib):
    """Every check runs before any CUDA call (this machine may have no GPU)."""
    buf = ctypes.create_string_buffer(1 << 16)
    p16 = (ctypes.addressof(buf) + 15) // 16 * 16
    ws_n = lib.triad_retrieve_ragged_workspace_bytes(77, 2, 10, 0)
    good = dict(qc=p16, qs=p16, Nq=77, codes=p16, scales=p16, meta=p16, info=p16, n_slots=2, n_cap=10, D=512, T=p16,
                direction=0, scores=p16, ws=p16, ws_bytes=ws_n)

    def call(**kw):
        a = dict(good, **kw)
        return lib.triad_retrieve_scores_ragged_e4m3(a["qc"], a["qs"], a["Nq"], a["codes"], a["scales"], a["meta"],
                                                     a["info"], a["n_slots"], a["n_cap"], a["D"], a["T"],
                                                     a["direction"], a["scores"], a["ws"], a["ws_bytes"], None)

    for name in ("qc", "qs", "codes", "scales", "meta", "info", "T", "scores", "ws"):
        assert call(**{name: None}) == -1, name                                   # TRIAD_ERR_BAD_ARG
    for d in (-1, 2, 5):
        assert call(direction=d) == -1
    for kw in (dict(Nq=0), dict(Nq=65536), dict(n_slots=0), dict(n_cap=1), dict(n_cap=2 * 256 + 1), dict(D=0)):
        assert call(**kw) == -2, kw                                               # TRIAD_ERR_BAD_SHAPE
    for D in (64, 192, 320, 640):                                                 # bf16 takes 64 and 192, e4m3 not
        assert call(D=D) == -7, D                                                 # TRIAD_ERR_UNSUPPORTED
    for kw in (dict(qc=p16 + 8), dict(codes=p16 + 8), dict(ws=p16 + 8), dict(meta=p16 + 4), dict(info=p16 + 4),
               dict(qs=p16 + 2), dict(scales=p16 + 2), dict(scores=p16 + 2)):
        assert call(**kw) == -3, kw                                               # TRIAD_ERR_ALIGNMENT
    assert call(ws_bytes=ws_n - 1) == -4                                          # TRIAD_ERR_WORKSPACE
    assert call(direction=1, ws_bytes=lib.triad_retrieve_ragged_workspace_bytes(77, 2, 10, 1) - 1) == -4


def _gallery(lens, D, fp8):
    meta, info = ragged_plan(lens)
    n = meta.shape[0] * SLOT
    if fp8:
        return RaggedGallery(torch.zeros(n, D, dtype=torch.uint8).view(torch.float8_e4m3fn), torch.from_numpy(meta),
                             torch.from_numpy(info), np.array(lens, np.int32), torch.arange(n, dtype=torch.float32))
    return RaggedGallery(torch.zeros(n, D, dtype=torch.bfloat16), torch.from_numpy(meta), torch.from_numpy(info),
                         np.array(lens, np.int32))


def test_fp8_storage_validation(lib):
    for D in (64, 192, 640, 1024):
        with pytest.raises(ValueError):
            RaggedGallery.from_list([torch.zeros(3, D), torch.zeros(5, D)], fp8=True)
        with pytest.raises(ValueError):
            RaggedGallery.from_padded(torch.zeros(2, 7, D), torch.ones(2, 7), fp8=True)
    bf, f8a, f8b = _gallery([100, 200], 128, False), _gallery([300 - 256 + 1, 7], 128, True), _gallery([256, 3], 128, True)
    assert bf.scales is None and RaggedGallery.cat([bf, bf]).scales is None
    with pytest.raises(ValueError):
        RaggedGallery.cat([bf, f8a])
    with pytest.raises(ValueError):
        RaggedGallery.cat([f8a, bf])
    j = RaggedGallery.cat([f8a, f8b])
    assert j.slots.dtype == torch.float8_e4m3fn and j.n_slots == 1 + 2 and len(j) == 4
    assert torch.equal(j.scales, torch.cat([f8a.scales, f8b.scales]))
    assert f8a.nbytes == SLOT * 128 + 4 * SLOT + 20 * 4 + 2 * 2 * 4
    assert j.nbytes == f8a.nbytes + f8b.nbytes
    assert bf.nbytes == 2 * SLOT * 128 * 2 + 2 * 20 * 4 + 2 * 2 * 4
