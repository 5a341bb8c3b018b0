"""CPU tier of the ragged caption gallery: the slot plan (triad_ragged_plan) against a greedy plan restated here, and
the argument checks of the new C entry points, which must reject bad arguments before any CUDA call."""
import ctypes

import numpy as np
import pytest

from triad_b200 import _lib, build

SLOT = 256


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _lib.load()


def greedy_plan(lengths):
    """(slots, info): slots = list of [first caption, count, used, starts (set of rows), ends (set of rows)],
    info[c] = (first row, length).  Greedy in order; a caption that does not fit starts a new slot."""
    slots, info = [], []
    for c, n in enumerate(lengths):
        if not slots or slots[-1][2] + n > SLOT:
            slots.append([c, 0, 0, set(), set()])
        s = slots[-1]
        off = s[2]
        s[1] += 1
        s[3].add(off)
        s[4].add(off + n - 1)
        s[2] += n
        info.append(((len(slots) - 1) * SLOT + off, n))
    return slots, info


def mask_words(rows):
    w = np.zeros(8, dtype=np.uint32)
    for r in rows:
        w[r // 32] |= np.uint32(1 << (r % 32))
    return w.view(np.int32)


def check_plan(lengths):
    from triad_b200.retrieval import ragged_plan
    meta, info = ragged_plan(lengths)
    slots, ref_info = greedy_plan(list(lengths))
    assert meta.shape == (len(slots), 20)
    assert info.tolist() == [list(x) for x in ref_info]
    for k, s in enumerate(slots):
        assert meta[k, :4].tolist() == [s[0], s[1], s[2], 0], k
        assert (meta[k, 4:12] == mask_words(s[3])).all(), k
        assert (meta[k, 12:20] == mask_words(s[4])).all(), k
    return meta, info


@pytest.mark.parametrize("lengths", [
    [1], [256], [1] * 300, [256] * 3,
    [128, 128, 1],                  # a slot filled exactly, then a new one
    [200, 56, 57],                  # exactly full, then a fresh slot
    [200, 57],                      # one row too many: the second caption starts a new slot
    [255, 1, 1, 255, 2],
    [1, 256, 1],
    [31, 1, 32, 33, 64, 95],        # starts and ends on both sides of 32-row word boundaries
])
def test_plan_matches_greedy(lib, lengths):
    check_plan(lengths)


def test_plan_matches_greedy_random(lib):
    rng = np.random.default_rng(7)
    check_plan(rng.integers(8, 78, size=5000))           # cfg 3's caption lengths
    check_plan(rng.integers(1, 257, size=2000))


def test_plan_rejects_bad_lengths(lib):
    from triad_b200.retrieval import ragged_plan
    for bad in ([0], [5, 0, 3], [257], [4, 300], []):
        with pytest.raises(ValueError):
            ragged_plan(bad)
    meta = np.zeros((4, 20), np.int32)
    info = np.zeros((4, 2), np.int32)
    n = ctypes.c_int(-1)
    for bad in ([3, 0], [257, 1], [-1, 2]):
        lens = np.array(bad, np.int32)
        assert lib.triad_ragged_plan(lens.ctypes.data, len(bad), meta.ctypes.data, info.ctypes.data,
                                     ctypes.byref(n)) == -2                          # TRIAD_ERR_BAD_SHAPE
    lens = np.array([3], np.int32)
    assert lib.triad_ragged_plan(lens.ctypes.data, 0, meta.ctypes.data, info.ctypes.data, ctypes.byref(n)) == -2
    assert lib.triad_ragged_plan(None, 1, meta.ctypes.data, info.ctypes.data, ctypes.byref(n)) == -1
    assert lib.triad_ragged_plan(lens.ctypes.data, 1, None, info.ctypes.data, ctypes.byref(n)) == -1
    assert lib.triad_ragged_plan(lens.ctypes.data, 1, meta.ctypes.data, None, ctypes.byref(n)) == -1
    assert lib.triad_ragged_plan(lens.ctypes.data, 1, meta.ctypes.data, info.ctypes.data, None) == -1


def test_cat_of_partly_full_slots(lib):
    """cat = slot concat with offsets: the same metadata as the plan of each part, caption ids and rows shifted."""
    import torch
    from triad_b200.retrieval import RaggedGallery, ragged_plan
    parts = [[100, 100, 30], [7], [256, 200, 100]]          # every part's last slot partly full
    gs = []
    for lens in parts:
        meta, info = ragged_plan(lens)
        gs.append(RaggedGallery(torch.zeros(meta.shape[0] * SLOT, 64, dtype=torch.bfloat16), torch.from_numpy(meta),
                                torch.from_numpy(info), np.array(lens, np.int32)))
    g = RaggedGallery.cat(gs)
    assert len(g) == g.shape[0] == 7 and g.n_slots == 1 + 1 + 3 and g.slots.shape == (5 * SLOT, 64)
    # the whole plan would pack differently (7 would join the first slot): cat keeps each part's slots
    slots = []
    cap0 = slot0 = 0
    infos = []
    for lens in parts:
        s, info = greedy_plan(lens)
        for x in s:
            slots.append([x[0] + cap0] + x[1:])
        infos += [(r + slot0 * SLOT, n) for r, n in info]
        cap0 += len(lens)
        slot0 += len(s)
    meta = g.meta.numpy()
    for k, s in enumerate(slots):
        assert meta[k, :4].tolist() == [s[0], s[1], s[2], 0]
        assert (meta[k, 4:12] == mask_words(s[3])).all() and (meta[k, 12:20] == mask_words(s[4])).all()
    assert g.cap_info.numpy().tolist() == [list(x) for x in infos]
    assert g.nbytes == 5 * SLOT * 64 * 2 + 5 * 20 * 4 + 7 * 2 * 4


def test_scores_ragged_rejects_bad_arguments(lib):
    """Every check runs before any CUDA call (this machine may have no GPU)."""
    buf = ctypes.create_string_buffer(1 << 16)
    p = ctypes.addressof(buf)
    p16 = (p + 15) // 16 * 16
    ws_n = lib.triad_retrieve_ragged_workspace_bytes(77, 2, 10, 0)
    assert ws_n > 0 and lib.triad_retrieve_ragged_workspace_bytes(77, 2, 10, 1) > 0
    assert lib.triad_retrieve_ragged_workspace_bytes(77, 2, 10, 2) == 0
    assert lib.triad_retrieve_ragged_workspace_bytes(0, 2, 10, 0) == 0
    assert lib.triad_retrieve_ragged_workspace_bytes(77, 0, 10, 0) == 0
    assert lib.triad_retrieve_ragged_workspace_bytes(77, 2, 0, 0) == 0
    good = dict(q=p16, Nq=77, slots=p16, meta=p16, info=p16, n_slots=2, n_cap=10, D=512, T=p16, direction=0,
                scores=p16, ws=p16, ws_bytes=ws_n)

    def call(**kw):
        a = dict(good, **kw)
        return lib.triad_retrieve_scores_ragged(a["q"], a["Nq"], a["slots"], a["meta"], a["info"], a["n_slots"],
                                                a["n_cap"], a["D"], a["T"], a["direction"], a["scores"], a["ws"],
                                                a["ws_bytes"], None)

    for name in ("q", "slots", "meta", "info", "T", "scores", "ws"):
        assert call(**{name: None}) == -1, name                                   # TRIAD_ERR_BAD_ARG
    for d in (-1, 2, 5):
        assert call(direction=d) == -1
    for kw in (dict(Nq=0), dict(Nq=65536), dict(n_slots=0), dict(n_cap=1), dict(n_cap=2 * 256 + 1), dict(D=0)):
        assert call(**kw) == -2, kw                                               # TRIAD_ERR_BAD_SHAPE
    for D in (32, 96, 576):
        assert call(D=D) == -7, D                                                 # TRIAD_ERR_UNSUPPORTED
    assert call(q=p16 + 8) == -3 and call(slots=p16 + 8) == -3 and call(meta=p16 + 4) == -3   # TRIAD_ERR_ALIGNMENT
    assert call(ws_bytes=ws_n - 1) == -4                                          # TRIAD_ERR_WORKSPACE
    assert call(direction=1, ws_bytes=lib.triad_retrieve_ragged_workspace_bytes(77, 2, 10, 1) - 1) == -4


def test_pack_rejects_bad_arguments(lib):
    buf = ctypes.create_string_buffer(4096)
    p16 = (ctypes.addressof(buf) + 15) // 16 * 16

    def call(src=p16, dtype=1, src_rows=4, D=64, rowmap=p16, dst_rows=256, dst=p16):
        return lib.triad_ragged_pack(src, dtype, src_rows, D, rowmap, dst_rows, dst, None)

    assert call(src=None) == -1 and call(rowmap=None) == -1 and call(dst=None) == -1
    assert call(dtype=7) == -1
    assert call(src_rows=0) == -2 and call(dst_rows=100) == -2 and call(D=12) == -2 and call(D=0) == -2
    assert call(src=p16 + 2) == -3 and call(dst=p16 + 8) == -3 and call(rowmap=p16 + 2) == -3
