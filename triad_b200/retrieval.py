"""Retrieval use of the max-mean kernel: drop-ins for src/retrieval.py's aggregators
(:106-115, :190-198), recall@k (:117-144) and the two metric drivers (:146-188, :250-292).

The reference fills each N x N similarity matrix with a Python double loop — 10^6 iterations,
each an H2D copy, a matmul and an ``.item()``.  Here a whole matrix is a handful of launches of
the same forward kernel used for training (both directions are max-mean with the operands
swapped), and the rank of the diagonal is computed on the device.
"""
from __future__ import annotations

import ctypes
from collections import defaultdict
from typing import Dict, List, Sequence

import numpy as np
import torch

from . import _lib, ops
from ._lib import check


def _scores(q_feats: torch.Tensor, v_feats: torch.Tensor, temperature, direction: int) -> torch.Tensor:
    """scores[n] for one query (Nq,D) against a gallery (n,Nv,D); retrieval divides by T."""
    lib = _lib.load()
    q = q_feats.contiguous()
    gal = v_feats.contiguous() if v_feats.dim() == 3 else v_feats.contiguous().unsqueeze(0)
    if q.dtype != gal.dtype:
        gal = gal.to(q.dtype)
    n_img, Nv, D = gal.shape
    Nq = q.shape[0]
    dt = ops._dtype_code(q)
    T = ops.temperature_tensor(temperature, q.device)
    out = torch.empty(n_img, dtype=torch.float32, device=q.device)
    nws = lib.triad_retrieve_workspace_bytes(Nq, n_img, Nv, D, dt)
    with ops._on(q):
        ws = ops._Workspace.get(nws, q.device, "retrieve")
        check(lib.triad_retrieve_scores(q.data_ptr(), Nq, gal.data_ptr(), n_img, Nv, D, dt, T.data_ptr(), 1, direction,
                                        out.data_ptr(), ws.data_ptr(), ws.numel(), ops._stream(q.device)),
              "triad_retrieve_scores")
    return out


def aggregator_av_a2v(a_feats, v_feats, temperature) -> float:
    """mean over audio frames of max over patches of (a.v/T) — retrieval.py:106-110."""
    return _scores(a_feats, v_feats, temperature, 0).item()


def aggregator_av_v2a(a_feats, v_feats, temperature) -> float:
    """mean over patches of max over audio frames — retrieval.py:112-115."""
    return _scores(a_feats, v_feats, temperature, 1).item()


def aggregator_tv_t2v(t_feats, v_feats, temperature) -> float:
    """retrieval.py:190-193."""
    return _scores(t_feats, v_feats, temperature, 0).item()


def aggregator_tv_v2t(t_feats, v_feats, temperature) -> float:
    """retrieval.py:195-198."""
    return _scores(t_feats, v_feats, temperature, 1).item()


class Fp8Gallery:
    """A retrieval gallery stored as e4m3 codes with one fp32 scale per patch: about half the bytes of bf16.

    ``codes`` is ``torch.float8_e4m3fn [n_img, Nv, D]`` and ``scales`` fp32 ``[n_img, Nv]``; patch p of image n stands
    for ``scales[n, p] * codes[n, p, :]``.  Each patch row is quantized on its own (``triad_quantize_e4m3``:
    s = amax / 448, codes = e4m3(x / s) with saturation), so quantizing a slice of a gallery gives exactly that slice of
    the quantized gallery.  ``retrieve_topk`` and ``dist.sharded_retrieve_topk`` accept it in place of a bf16 tensor
    (direction 0 only).  D must be 128, 256, 384 or 512."""

    def __init__(self, codes: torch.Tensor, scales: torch.Tensor):
        if codes.dtype != torch.float8_e4m3fn or codes.dim() != 3:
            raise ValueError("Fp8Gallery: codes must be a float8_e4m3fn tensor [n_img, Nv, D]")
        n_img, Nv, D = codes.shape
        _check_fp8_shape(n_img, Nv, D)
        if scales.dtype != torch.float32 or tuple(scales.shape) != (n_img, Nv):
            raise ValueError(f"Fp8Gallery: scales must be float32 [{n_img}, {Nv}], got {scales.dtype} {tuple(scales.shape)}")
        if codes.device != scales.device or not codes.is_contiguous() or not scales.is_contiguous():
            raise ValueError("Fp8Gallery: codes and scales must be contiguous and on the same device")
        self.codes = codes
        self.scales = scales

    @classmethod
    def empty(cls, n_img: int, Nv: int, D: int, device="cuda") -> "Fp8Gallery":
        _check_fp8_shape(n_img, Nv, D)
        return cls(torch.empty(n_img, Nv, D, dtype=torch.float8_e4m3fn, device=device),
                   torch.empty(n_img, Nv, dtype=torch.float32, device=device))

    @property
    def shape(self):
        return tuple(self.codes.shape)

    @property
    def device(self) -> torch.device:
        return self.codes.device

    @property
    def nbytes(self) -> int:
        n_img, Nv, D = self.shape
        return n_img * Nv * D + 4 * n_img * Nv

    def __len__(self) -> int:
        return self.shape[0]

    def __getitem__(self, sl) -> "Fp8Gallery":
        """Images [start, stop) as a view (no copy): a contiguous shard of the gallery."""
        if not isinstance(sl, slice) or sl.step not in (None, 1):
            raise TypeError("Fp8Gallery: only contiguous slices of images are supported")
        return Fp8Gallery(self.codes[sl], self.scales[sl])

    def put(self, i0: int, feats: torch.Tensor) -> None:
        """Quantize the embedded images ``feats`` ([b, Nv, D] bf16 or fp32, on the gallery's device) into images
        [i0, i0 + b).  Lets a caller build a gallery larger than its bf16 form would fit, batch by batch."""
        n_img, Nv, D = self.shape
        if feats.dim() != 3 or tuple(feats.shape[1:]) != (Nv, D):
            raise ValueError(f"Fp8Gallery.put: feats must be [b, {Nv}, {D}], got {tuple(feats.shape)}")
        b = feats.shape[0]
        if not 0 <= i0 or i0 + b > n_img:
            raise IndexError(f"Fp8Gallery.put: images [{i0}, {i0 + b}) outside [0, {n_img})")
        if feats.device != self.device:
            raise ValueError("Fp8Gallery.put: feats must be on the gallery's device")
        if b == 0:
            return
        _quantize_rows(feats, self.codes[i0:i0 + b], self.scales[i0:i0 + b])


def _check_fp8_shape(n_img: int, Nv: int, D: int) -> None:
    if n_img < 1 or not 1 <= Nv <= 65535:
        raise ValueError(f"Fp8Gallery: need n_img >= 1 and 1 <= Nv <= 65535, got n_img={n_img}, Nv={Nv}")
    if D % 128 or not 128 <= D <= 512:
        raise ValueError(f"Fp8Gallery: D must be 128, 256, 384 or 512, got {D}")


def _quantize_rows(x: torch.Tensor, codes: torch.Tensor, scales: torch.Tensor) -> None:
    """triad_quantize_e4m3 of the rows of x (last dim D) into codes / scales of the same row count."""
    lib = _lib.load()
    x = x.contiguous()
    dt = ops._dtype_code(x)
    D = x.shape[-1]
    rows = x.numel() // D
    with ops._on(x):
        check(lib.triad_quantize_e4m3(x.data_ptr(), dt, rows, D, codes.data_ptr(), scales.data_ptr(), ops._stream(x.device)),
              "triad_quantize_e4m3")


def quantize_gallery(feats: torch.Tensor) -> Fp8Gallery:
    """Fp8Gallery of the embedded gallery ``feats`` ([n_img, Nv, D] bf16 or fp32)."""
    if feats.dim() != 3:
        raise ValueError(f"quantize_gallery: feats must be [n_img, Nv, D], got {tuple(feats.shape)}")
    g = Fp8Gallery.empty(*feats.shape, device=feats.device)
    g.put(0, feats)
    return g


def _scores_fp8(q_feats: torch.Tensor, gallery: Fp8Gallery, temperature, direction: int) -> torch.Tensor:
    """scores[n] of one query (Nq, D) against an e4m3 gallery: the query is quantized per token on the device, then
    scored with the tensor cores' kind::f8f6f4 MMA (triad_retrieve_scores_e4m3)."""
    if direction != 0:
        raise ValueError("an Fp8Gallery supports direction 0 (mean over query tokens of max over patches) only")
    n_img, Nv, D = gallery.shape
    if q_feats.dim() != 2 or q_feats.shape[1] != D:
        raise ValueError(f"query must be [Nq, {D}], got {tuple(q_feats.shape)}")
    lib = _lib.load()
    q = q_feats.contiguous()
    Nq = q.shape[0]
    dev = gallery.device
    q_codes = torch.empty(Nq, D, dtype=torch.uint8, device=dev)
    q_scales = torch.empty(Nq, dtype=torch.float32, device=dev)
    _quantize_rows(q, q_codes, q_scales)
    T = ops.temperature_tensor(temperature, dev)
    out = torch.empty(n_img, dtype=torch.float32, device=dev)
    nws = lib.triad_retrieve_e4m3_workspace_bytes(Nq, n_img, Nv, D)
    with ops._on(out):
        ws = ops._Workspace.get(nws, dev, "retrieve_e4m3")
        check(lib.triad_retrieve_scores_e4m3(q_codes.data_ptr(), q_scales.data_ptr(), Nq, gallery.codes.data_ptr(),
                                             gallery.scales.data_ptr(), n_img, Nv, D, T.data_ptr(), out.data_ptr(),
                                             ws.data_ptr(), ws.numel(), ops._stream(dev)), "triad_retrieve_scores_e4m3")
    return out


SLOT_ROWS = 256           # rows of one slot of a RaggedGallery, and the longest caption it stores
_SLOT_META_INTS = 20      # triad_ragged_plan: first caption, count, used rows, 0, start mask [8], end mask [8]


def ragged_plan(lengths) -> tuple:
    """(slot_meta int32 [n_slots, 20], cap_info int32 [n_cap, 2]) of captions with these lengths, on the host
    (triad_ragged_plan): greedy in order, a caption that does not fit in the rest of the current 256-row slot starts
    a new one.  cap_info[c] = (first row = slot * 256 + offset, length).  Lengths must be 1..256."""
    lens = np.ascontiguousarray(np.asarray(lengths, dtype=np.int64).reshape(-1))
    if lens.size == 0:
        raise ValueError("RaggedGallery: need at least one caption")
    if lens.min() < 1 or lens.max() > SLOT_ROWS:
        raise ValueError(f"RaggedGallery: caption lengths must be 1..{SLOT_ROWS}, got {int(lens.min())}..{int(lens.max())}")
    lens = lens.astype(np.int32)
    n = lens.size
    meta = np.zeros((n, _SLOT_META_INTS), dtype=np.int32)
    info = np.zeros((n, 2), dtype=np.int32)
    n_slots = ctypes.c_int(0)
    check(_lib.load().triad_ragged_plan(lens.ctypes.data, n, meta.ctypes.data, info.ctypes.data, ctypes.byref(n_slots)),
          "triad_ragged_plan")
    return meta[:n_slots.value].copy(), info


class RaggedGallery:
    """A gallery of items with different token counts (captions truncated to their valid tokens), stored without
    padding: the token rows of whole captions in 256-row slots, ``slots`` [n_slots * 256, D].

    Captions are placed greedily in order; one that does not fit in the rest of the current slot starts a new slot,
    so no caption straddles a slot, and a slot's rows after its last caption are zero.  ``meta`` (int32
    [n_slots, 20]) and ``cap_info`` (int32 [n_cap, 2]) describe the layout (``ragged_plan``).  Caption lengths must
    be 1..256.

    Two storages (``fp8`` of the builders):
    - bf16 (default): ``slots`` bf16; fp32 features are rounded to bf16 when the gallery is built; ``scales`` is None.
    - e4m3: ``slots`` float8_e4m3fn and ``scales`` fp32 [n_slots * 256], one per slot row, each row quantized on its
      own from the features in their own dtype (``triad_ragged_pack_e4m3``, bit-equal to ``triad_quantize_e4m3`` of
      that row; fp32 is not rounded to bf16 first).  Rows after a slot's last caption have scale 0 and zero codes.
      About half the bytes; D must be 128, 256, 384 or 512.

    ``retrieve_topk`` and ``dist.sharded_retrieve_topk`` accept it in place of a dense tensor, in both directions;
    ids are caption numbers.  ``len()`` and ``shape[0]`` are the caption count; ``shape`` is (n_cap, D)."""

    def __init__(self, slots: torch.Tensor, meta: torch.Tensor, cap_info: torch.Tensor, lengths: np.ndarray,
                 scales: torch.Tensor = None):
        self.slots = slots
        self.meta = meta
        self.cap_info = cap_info
        self.lengths = lengths
        self.scales = scales

    @classmethod
    def _build(cls, src: torch.Tensor, src_rows: np.ndarray, lengths: np.ndarray, fp8: bool) -> "RaggedGallery":
        """Caption c is rows src_rows[sum(lengths[:c]) : ...] of src ([rows, D] fp32 or bf16, on the device)."""
        D = src.shape[1]
        if fp8 and (D % 128 or not 128 <= D <= 512):
            raise ValueError(f"RaggedGallery: an fp8 gallery needs D of 128, 256, 384 or 512, got {D}")
        meta, info = ragged_plan(lengths)
        n_slots = meta.shape[0]
        dev = src.device
        rowmap = np.full(n_slots * SLOT_ROWS, -1, dtype=np.int32)
        firsts = np.repeat(info[:, 0].astype(np.int64), lengths)
        within = np.arange(int(lengths.sum()), dtype=np.int64) - np.repeat(np.cumsum(lengths) - lengths, lengths)
        rowmap[firsts + within] = src_rows
        src = src.contiguous()
        if src.dtype not in (torch.float32, torch.bfloat16):
            src = src.float()
        rm = torch.from_numpy(rowmap).to(dev)
        lib = _lib.load()
        scales = None
        with ops._on(src):
            if fp8:
                slots = torch.empty(n_slots * SLOT_ROWS, D, dtype=torch.float8_e4m3fn, device=dev)
                scales = torch.empty(n_slots * SLOT_ROWS, dtype=torch.float32, device=dev)
                check(lib.triad_ragged_pack_e4m3(src.data_ptr(), ops._dtype_code(src), src.shape[0], D, rm.data_ptr(),
                                                 slots.shape[0], slots.data_ptr(), scales.data_ptr(), ops._stream(dev)),
                      "triad_ragged_pack_e4m3")
            else:
                slots = torch.empty(n_slots * SLOT_ROWS, D, dtype=torch.bfloat16, device=dev)
                check(lib.triad_ragged_pack(src.data_ptr(), ops._dtype_code(src), src.shape[0], D, rm.data_ptr(),
                                            slots.shape[0], slots.data_ptr(), ops._stream(dev)), "triad_ragged_pack")
        return cls(slots, torch.from_numpy(meta).to(dev), torch.from_numpy(info).to(dev), lengths.astype(np.int32),
                   scales)

    @classmethod
    def from_padded(cls, feats: torch.Tensor, attention_mask, fp8: bool = False) -> "RaggedGallery":
        """Captions from the text embedder's output: feats [b, L, D] and attention_mask [b, L]; caption i keeps the
        rows whose mask is non-zero, in order (the reference's truncation for right-padded masks).  ``fp8`` stores
        e4m3 codes with one scale per row instead of bf16."""
        if feats.dim() != 3:
            raise ValueError(f"RaggedGallery.from_padded: feats must be [b, L, D], got {tuple(feats.shape)}")
        b, L, D = feats.shape
        mask = (torch.as_tensor(attention_mask).detach().to("cpu").numpy() != 0)
        if mask.shape != (b, L):
            raise ValueError(f"RaggedGallery.from_padded: attention_mask must be [{b}, {L}], got {mask.shape}")
        lengths = mask.sum(axis=1)
        src_rows = np.flatnonzero(mask.reshape(-1)).astype(np.int32)
        return cls._build(feats.reshape(b * L, D), src_rows, lengths, fp8)

    @classmethod
    def from_list(cls, feats: Sequence[torch.Tensor], fp8: bool = False) -> "RaggedGallery":
        """Captions from a list of [L_i, D] tensors (what the reference's embed_tv_subset returns).  ``fp8`` stores
        e4m3 codes with one scale per row instead of bf16."""
        if len(feats) == 0:
            raise ValueError("RaggedGallery.from_list: need at least one caption")
        if any(t.dim() != 2 for t in feats) or len({t.shape[1] for t in feats}) != 1:
            raise ValueError("RaggedGallery.from_list: captions must be [L_i, D] with one D")
        lengths = np.array([t.shape[0] for t in feats], dtype=np.int64)
        src = torch.cat([t.to(feats[0].dtype) for t in feats])
        return cls._build(src, np.arange(src.shape[0], dtype=np.int32), lengths, fp8)

    @classmethod
    def cat(cls, galleries: Sequence["RaggedGallery"]) -> "RaggedGallery":
        """The captions of several galleries, in order (caption ids continue from one gallery to the next).  Slots
        are independent, so this concatenates slot arrays: a large gallery can be built batch by batch."""
        if len(galleries) == 0:
            raise ValueError("RaggedGallery.cat: need at least one gallery")
        D, dev = galleries[0].shape[1], galleries[0].device
        if any(g.shape[1] != D or g.device != dev for g in galleries):
            raise ValueError("RaggedGallery.cat: galleries must share D and device")
        if len({g.slots.dtype for g in galleries}) != 1:
            raise ValueError("RaggedGallery.cat: galleries must share their storage (all bf16 or all fp8)")
        metas, infos = [], []
        cap_off = slot_off = 0
        for g in galleries:
            m = g.meta.clone()
            m[:, 0] += cap_off
            i = g.cap_info.clone()
            i[:, 0] += slot_off * SLOT_ROWS
            metas.append(m)
            infos.append(i)
            cap_off += len(g)
            slot_off += g.n_slots
        scales = None if galleries[0].scales is None else torch.cat([g.scales for g in galleries])
        return cls(torch.cat([g.slots for g in galleries]), torch.cat(metas), torch.cat(infos),
                   np.concatenate([g.lengths for g in galleries]), scales)

    @property
    def n_slots(self) -> int:
        return self.meta.shape[0]

    @property
    def shape(self):
        return (self.cap_info.shape[0], self.slots.shape[1])

    @property
    def device(self) -> torch.device:
        return self.slots.device

    @property
    def nbytes(self) -> int:
        scale_bytes = 0 if self.scales is None else self.scales.numel() * 4
        return (self.slots.numel() * self.slots.element_size() + scale_bytes + self.meta.numel() * 4
                + self.cap_info.numel() * 4)

    def __len__(self) -> int:
        return self.cap_info.shape[0]


def _scores_ragged(q_feats: torch.Tensor, gallery: RaggedGallery, temperature, direction: int) -> torch.Tensor:
    """scores[c] of one query (Nq, D) against every caption of a ragged gallery: a bf16 gallery rounds the query to
    bf16 (triad_retrieve_scores_ragged), an fp8 one quantizes it per token on the device
    (triad_retrieve_scores_ragged_e4m3)."""
    n_cap, D = gallery.shape
    if q_feats.dim() != 2 or q_feats.shape[1] != D:
        raise ValueError(f"query must be [Nq, {D}], got {tuple(q_feats.shape)}")
    if direction not in (0, 1):
        raise ValueError(f"direction must be 0 or 1, got {direction}")
    lib = _lib.load()
    dev = gallery.device
    Nq = q_feats.shape[0]
    T = ops.temperature_tensor(temperature, dev)
    out = torch.empty(n_cap, dtype=torch.float32, device=dev)
    nws = lib.triad_retrieve_ragged_workspace_bytes(Nq, gallery.n_slots, n_cap, direction)
    if gallery.scales is not None:
        q = q_feats.to(device=dev).contiguous()
        q_codes = torch.empty(Nq, D, dtype=torch.uint8, device=dev)
        q_scales = torch.empty(Nq, dtype=torch.float32, device=dev)
        _quantize_rows(q, q_codes, q_scales)
        with ops._on(out):
            ws = ops._Workspace.get(nws, dev, "retrieve_ragged")
            check(lib.triad_retrieve_scores_ragged_e4m3(
                q_codes.data_ptr(), q_scales.data_ptr(), Nq, gallery.slots.data_ptr(), gallery.scales.data_ptr(),
                gallery.meta.data_ptr(), gallery.cap_info.data_ptr(), gallery.n_slots, n_cap, D, T.data_ptr(), direction,
                out.data_ptr(), ws.data_ptr(), ws.numel(), ops._stream(dev)), "triad_retrieve_scores_ragged_e4m3")
        return out
    q = q_feats.to(device=dev, dtype=torch.bfloat16).contiguous()
    with ops._on(out):
        ws = ops._Workspace.get(nws, dev, "retrieve_ragged")
        check(lib.triad_retrieve_scores_ragged(q.data_ptr(), Nq, gallery.slots.data_ptr(), gallery.meta.data_ptr(),
                                               gallery.cap_info.data_ptr(), gallery.n_slots, n_cap, D, T.data_ptr(),
                                               direction, out.data_ptr(), ws.data_ptr(), ws.numel(), ops._stream(dev)),
              "triad_retrieve_scores_ragged")
    return out


def retrieve_topk(q_feats: torch.Tensor, gallery, temperature, k: int, direction: int = 0):
    """Top-k gallery items for one query (BASELINE cfg 5): (scores fp32 [k], ids int32 [k]).

    ``gallery`` is an embedding tensor [n_img, Nv, D], an ``Fp8Gallery`` (e4m3 codes with per-patch scales; the
    query is then quantized per token in the same call, and only direction 0 is supported) or a ``RaggedGallery``
    (captions of different lengths, both directions; the query is rounded to bf16 for a bf16 gallery and quantized
    per token in the same call for an fp8 one)."""
    if isinstance(gallery, Fp8Gallery):
        s = _scores_fp8(q_feats, gallery, temperature, direction)
    elif isinstance(gallery, RaggedGallery):
        s = _scores_ragged(q_feats, gallery, temperature, direction)
    else:
        s = _scores(q_feats, gallery, temperature, direction)
    return _topk(s, k)


def _topk(s: torch.Tensor, k: int):
    """(scores, ids) of the k largest entries of s, ties to the lower id (triad_topk)."""
    lib = _lib.load()
    n = s.numel()
    out_s = torch.empty(k, dtype=torch.float32, device=s.device)
    out_i = torch.empty(k, dtype=torch.int32, device=s.device)
    nws = lib.triad_topk_workspace_bytes(n, k)
    with ops._on(s):
        ws = ops._Workspace.get(nws, s.device, "topk")
        check(lib.triad_topk(s.data_ptr(), n, k, out_s.data_ptr(), out_i.data_ptr(), ws.data_ptr(), ws.numel(),
                             ops._stream(s.device)), "triad_topk")
    return out_s, out_i


def pairwise_similarity(q_list: Sequence[torch.Tensor], v_list: Sequence[torch.Tensor], temperature,
                        direction: int = 0, device="cuda") -> torch.Tensor:
    """sim[i,j] = aggregator(q_list[i], v_list[j]) for every pair, on the device.

    direction 0: mean_q max_v (a2v / t2v); direction 1: mean_v max_q (v2a / v2t).  Items may have
    different lengths (text is truncated to its valid tokens, retrieval.py:243-244): they are
    grouped by length and each (query-length, gallery-length) group is one forward launch."""
    T = ops.temperature_tensor(temperature, torch.device(device))
    rows, cols = (q_list, v_list) if direction == 0 else (v_list, q_list)
    n_r, n_c = len(rows), len(cols)
    sim = torch.empty(n_r, n_c, dtype=torch.float32, device=device)
    by_len_r: Dict[int, List[int]] = defaultdict(list)
    by_len_c: Dict[int, List[int]] = defaultdict(list)
    for i, t in enumerate(rows):
        by_len_r[t.shape[0]].append(i)
    for j, t in enumerate(cols):
        by_len_c[t.shape[0]].append(j)
    for nr, ri in by_len_r.items():
        R = torch.stack([rows[i] for i in ri]).to(device)
        scale = ops.row_scale(None, R.shape[0], nr, R.device)
        for nc, ci in by_len_c.items():
            Cm = torch.stack([cols[j] for j in ci]).to(device=device, dtype=R.dtype)
            clip, _ = ops.maxmean_fwd(R, Cm, scale, T, want_idx=False, flags=_lib.FWD_DIVIDE_BY_T)
            sim[torch.tensor(ri, device=device)[:, None], torch.tensor(ci, device=device)[None, :]] = clip
    return sim if direction == 0 else sim.t().contiguous()


def compute_recall_at_k(sim_matrix) -> Dict[str, float]:
    """R@1/5/10/20 with the diagonal as ground truth — retrieval.py:117-144.  Accepts the numpy
    array the reference passes or a CUDA tensor; ranks are computed on the device."""
    lib = _lib.load()
    if isinstance(sim_matrix, np.ndarray):
        sim = torch.from_numpy(np.ascontiguousarray(sim_matrix, dtype=np.float32)).cuda()
    else:
        sim = sim_matrix.detach().float().contiguous()
    N = sim.shape[0]
    ranks = torch.empty(N, dtype=torch.int32, device=sim.device)
    with ops._on(sim):
        check(lib.triad_diag_ranks(sim.data_ptr(), N, ranks.data_ptr(), ops._stream(sim.device)), "triad_diag_ranks")
    r = ranks.cpu().numpy()
    return {"r1": float(np.mean(r < 1)), "r5": float(np.mean(r < 5)),
            "r10": float(np.mean(r < 10)), "r20": float(np.mean(r < 20))}


def _metrics(q_list, v_list, temperature, device, tag_q: str, tag_v: str) -> Dict[str, float]:
    fwd = compute_recall_at_k(pairwise_similarity(q_list, v_list, temperature, 0, device))
    # the reference's V->Q matrix is indexed [image i, query j] (retrieval.py:170-175)
    rev = compute_recall_at_k(pairwise_similarity(q_list, v_list, temperature, 1, device).t().contiguous())
    out = {}
    for k in (1, 5, 10, 20):
        out[f"{tag_q}->{tag_v}_r{k}"] = fwd[f"r{k}"]
    for k in (1, 5, 10, 20):
        out[f"{tag_v}->{tag_q}_r{k}"] = rev[f"r{k}"]
    return out


def metrics_from_features(q_list, v_list, temperature, device="cuda", kind: str = "av") -> Dict[str, float]:
    """The eight recalls of retrieval.py:177-187 / :281-291 from already-embedded items."""
    return _metrics(q_list, v_list, temperature, device, "A" if kind == "av" else "T", "V")


def compute_av_retrieval_metrics(model, dataset, subset_file, device="cuda"):
    """retrieval.py:146-188 with the 2 x 10^6-iteration aggregator loops replaced.  Subset selection
    and embedding are the caller-side steps of the reference (retrieval.py:9-30, :32-104), kept as is:
    pass the reference module's helpers through ``model``/``dataset`` unchanged."""
    import importlib
    ref = importlib.import_module("retrieval")      # the reference's own module, for its embed helpers
    indices = ref.select_subset_indices(dataset, subset_file, subset_size=1000)
    audio_feats, video_feats, _ = ref.embed_av_subset(model, dataset, indices, device=device, batch_size=8)
    return metrics_from_features(audio_feats, video_feats, model.temperature.item(), device, "av")


def compute_tv_retrieval_metrics(model, dataset, subset_file, device="cuda"):
    """retrieval.py:250-292, see compute_av_retrieval_metrics."""
    import importlib
    ref = importlib.import_module("retrieval")
    indices = ref.select_subset_indices(dataset, subset_file, subset_size=1000)
    text_feats, image_feats = ref.embed_tv_subset(model, dataset, indices, device=device, batch_size=8)
    return metrics_from_features(text_feats, image_feats, model.temperature.item(), device, "tv")
