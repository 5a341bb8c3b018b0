"""CPU tier: the e4m3 retrieval gallery's argument checks and host logic, without a GPU.

Every check of ``triad_quantize_e4m3``, ``triad_retrieve_e4m3_workspace_bytes`` and ``triad_retrieve_scores_e4m3``
(null pointers, alignment, shapes, workspace size) runs before the first CUDA call, so a wrong argument is reported
the same way on a machine without a device.  The pointers below are never dereferenced.  Also: the argmax buffer the
forwards allocate has its per-query padding defined (0)."""
import pytest
import torch

from triad_b200 import _lib, retrieval as R

OK, BAD_ARG, BAD_SHAPE, ALIGN, WS, UNSUP = 0, -1, -2, -3, -4, -7
P = 0x7f0000000000          # a 16-byte aligned stand-in for a device pointer
BIG = 1 << 40


@pytest.fixture(scope="module")
def lib():
    return _lib.load()


def _scores_call(lib, qc=P, qs=P, Nq=77, gc=P, gs=P, n=1000, Nv=1024, D=512, T=P, out=P, ws=P, ws_bytes=BIG):
    return lib.triad_retrieve_scores_e4m3(qc, qs, Nq, gc, gs, n, Nv, D, T, out, ws, ws_bytes, None)


def test_retrieve_e4m3_rejects_null_pointers(lib):
    for name in ("qc", "qs", "gc", "gs", "T", "out", "ws"):
        assert _scores_call(lib, **{name: None}) == BAD_ARG, name


def test_retrieve_e4m3_rejects_bad_shapes(lib):
    assert _scores_call(lib, Nq=0) == BAD_SHAPE
    assert _scores_call(lib, n=0) == BAD_SHAPE
    assert _scores_call(lib, Nv=0) == BAD_SHAPE
    assert _scores_call(lib, Nv=65536) == BAD_SHAPE
    for D in (64, 192, 320, 640, 1024):                  # D % 128 != 0 or D > 512
        assert _scores_call(lib, D=D) == UNSUP, D


def test_retrieve_e4m3_rejects_misaligned_pointers(lib):
    for name in ("qc", "gc", "ws"):                       # 16 bytes (TMA / workspace)
        assert _scores_call(lib, **{name: P + 8}) == ALIGN, name
    for name in ("qs", "gs", "out"):                      # 4 bytes
        assert _scores_call(lib, **{name: P + 2}) == ALIGN, name


def test_retrieve_e4m3_workspace(lib):
    need = lib.triad_retrieve_e4m3_workspace_bytes(77, 1000, 1024, 512)
    assert need > 0
    assert lib.triad_retrieve_e4m3_workspace_bytes(0, 1000, 1024, 512) == 0
    assert lib.triad_retrieve_e4m3_workspace_bytes(77, 0, 1024, 512) == 0
    assert lib.triad_retrieve_e4m3_workspace_bytes(77, 2000, 1024, 512) > need
    # query-sized, not gallery-sized: a few dozen bytes per image
    assert need < 64 * 1000 + 4096
    assert _scores_call(lib, ws_bytes=need - 1) == WS


def test_quantize_e4m3_rejects_bad_arguments(lib):
    q = lambda x=P, dt=1, rows=10, D=512, c=P, s=P: lib.triad_quantize_e4m3(x, dt, rows, D, c, s, None)  # noqa: E731
    assert q(x=None) == BAD_ARG and q(c=None) == BAD_ARG and q(s=None) == BAD_ARG
    assert q(dt=2) == BAD_ARG
    assert q(rows=0) == BAD_SHAPE and q(D=0) == BAD_SHAPE and q(D=24) == BAD_SHAPE and q(D=528) == BAD_SHAPE
    assert q(x=P + 8) == ALIGN and q(c=P + 8) == ALIGN and q(s=P + 2) == ALIGN


def test_fp8_gallery_host_logic():
    g = R.Fp8Gallery.empty(5, 13, 256, device="cpu")
    assert g.shape == (5, 13, 256) and len(g) == 5
    assert g.nbytes == 5 * 13 * 256 + 4 * 5 * 13
    assert g.codes.dtype == torch.float8_e4m3fn and g.scales.dtype == torch.float32
    s = g[1:4]
    assert s.shape == (3, 13, 256) and s.codes.data_ptr() == g.codes[1].data_ptr()
    with pytest.raises(TypeError):
        g[::2]
    for bad in ((0, 13, 256), (5, 0, 256), (5, 65536, 256), (5, 13, 64), (5, 13, 640), (5, 13, 200)):
        with pytest.raises(ValueError):
            R.Fp8Gallery.empty(*bad, device="cpu")
    feats = torch.zeros(2, 13, 256)
    for i0 in (-1, 4, 5):                                 # [i0, i0 + 2) must lie inside [0, 5)
        with pytest.raises(IndexError):
            g.put(i0, feats)
    with pytest.raises(ValueError):
        g.put(0, torch.zeros(2, 12, 256))
    with pytest.raises(ValueError):
        g.put(0, torch.zeros(2, 13, 128))
    with pytest.raises(ValueError):
        R.Fp8Gallery(torch.zeros(5, 13, 256, dtype=torch.uint8), torch.zeros(5, 13))
    with pytest.raises(ValueError):
        R.Fp8Gallery(g.codes, torch.zeros(5, 12))


def test_fp8_gallery_direction_1_raises():
    g = R.Fp8Gallery.empty(5, 13, 256, device="cpu")
    with pytest.raises(ValueError, match="direction 0"):
        R.retrieve_topk(torch.zeros(7, 256), g, 1.5, 3, direction=1)


@pytest.mark.parametrize("Nq,Nv", [(250, 256), (77, 1024), (64, 200)])
def test_argmax_buffer_padding_is_defined(Nq, Nv):
    """The forward's argmax buffer comes with its per-query padding (a >= Nq, never written by the kernels) set to 0,
    so buffers of two forwards of the same inputs compare equal whatever memory they were allocated from."""
    from triad_b200 import ops
    idx = ops.idx_buffer(3, 5, Nq, Nv, "cpu")
    nqp = ops.nq_padded(Nq)
    assert idx.shape == (3, 5 * nqp) and idx.dtype == ops.idx_dtype(Nv)
    assert (idx.view(3, 5, nqp)[:, :, Nq:] == 0).all()
