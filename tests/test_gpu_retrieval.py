"""GPU tier: the retrieval path (BASELINE cfg 5 and the recall metrics) against plain fp64 references, element by element.

A. ``triad_retrieve_scores`` in both directions, on galleries sized so that the forward takes each path a one-query
   retrieval can take: the SIMT kernels, the tcgen05 kernel with one and with two CTAs, in the default tile order and
   in the retrieval order (``sync = 0``, chunks of C = 1..64 images per cluster), with and without 256-patch sub-tiles.
B. ``retrieve_topk`` on those scores: its order against the kernel's own scores (exact) and against the fp64 scores
   (exact on the planted images, certified in the random tail).
C. ``triad_topk`` on synthetic vectors from one to 2^22 + 3 entries: ties across chunks, signed zeros, infinities,
   subnormals.
D. ``triad_diag_ranks`` / ``compute_recall_at_k``: ties at the diagonal, infinities, signed zeros, NaN.
E. ``triad_similarity_matrix``.

Tolerance of a score (A).  With e_ap = <q_a, v_p> / T exact (fp64 of the same bf16 / fp32 inputs), the kernels
compute S_ap = bf16(bf16(acc_ap) * fp32(1/T)) for bf16 inputs and fp32(acc_ap * fp32(1/T)) for fp32 inputs
(triad_round.h, round_sim with the reciprocal temperature).  acc_ap is an fp32 sum of D products,
|acc_ap - <q_a, v_p>| <= D 2^-23 |q_a| |v_p| (tensor-core accumulation is allowed 2 ulps per step).  A bf16 rounding
moves a value by at most 2^-8 of itself (8 significant bits), an fp32 one by 2^-24, so
    |S_ap - e_ap| <= rel |e_ap| + (1 + 2^-6) D 2^-23 |q_a| |v_p| / T,
    rel = 2^-7 + 2^-15 (two bf16 roundings, the reciprocal and the product) or 2^-23 (fp32).
Max over patches is 1-Lipschitz in the max norm, so |max_p S_ap - max_p e_ap| <= max_p of that bound, and the mean
over K rows (K = Nq in direction 0, Nv in direction 1) adds its weight 1/K and an fp32 sum, at most
(K + 3) 2^-24 mean_a max_p |e_ap| (1 + 2^-6).  Hence, per score n,
    tol_n = rel A_n + (1 + 2^-6) (D 2^-23 B_n / T + (K + 3) 2^-24 A_n),
    A_n = mean_a max_p |e_ap|,   B_n = mean_a max_p |q_a| |v_np|
(a and p swap roles in direction 1).  Each of the two bf16 roundings can take up to 2^-8, hence 2^-7 together.

Galleries.  Most images are random unit-norm patches.  A few are planted: every patch p of a planted image has cosine
c_n with query token p mod Nq (the noise is made orthogonal to that token), for graded levels c_n, so their fp64
scores are far apart.  Each case asserts its own premise: the smallest fp64 gap between planted scores is more than
10x the largest tolerance among them, so a shifted or swapped score cannot hide under the tolerance.  With
rel = 2^-7 that needs level steps of 0.085 (bf16), so a bf16 gallery holds as many levels as fit above its best
random image (at least 4, at most 12); fp32 galleries hold up to 32.  Planted images sit at id 0, on both sides of a C-chunk boundary and of
the 4096-id boundary of the top-k chunks, and at the last id; two of them are exact copies of others, in different
C-chunks (and different 4096-chunks when the gallery has two), whose scores must be bit-equal and whose top-k order
must follow their ids.
"""
import math

import numpy as np
import pytest
import torch

from triad_b200 import _lib, ops, retrieval as R
from triad_b200._lib import TriadError, check

pytestmark = pytest.mark.gpu

_SMS = torch.cuda.get_device_properties(0).multi_processor_count if torch.cuda.is_available() else 148
_MiB = 1 << 20
_TOPK_CHUNK = 4096


# ----------------------------------------------------------------------------------------------------------------
# which path a call takes: fwd_impl (capi.cu) and launch_maxmean_tc (maxmean_tc.cu), triad_topk (retrieve.cu)
# ----------------------------------------------------------------------------------------------------------------
def _fwd_path(dtype, M, Bv, Nv, D, sms=_SMS):
    """(kernel, tile order, C, sub-tiles) of the forward for M rows against Bv images of Nv patches."""
    if dtype == torch.float32:
        return "simt-f32", None, None, False
    if D % 64 or not 64 <= D <= 512:
        return "simt-bf16", None, None, False
    cta = 1 if M <= 128 else 2
    n_m = -(-M // (128 * cta))
    img = Nv * D * 2
    clusters = sms // cta
    order, C = "default", Bv
    if Bv * img > 48 * _MiB:
        c16 = max(1, 16 * _MiB // img)
        if n_m * c16 >= 4 * clusters:
            order, C = "sync", min(c16, Bv)
        else:
            order, C = "retrieval", min(max(1, min(64, 48 * _MiB // (clusters * img))), Bv)
    return f"tc{cta}", order, C, Nv > 256


def _topk_levels(n, k):
    """Number of chunk-sort passes triad_topk makes."""
    cur, levels = n, 0
    while True:
        nchunk = -(-cur // _TOPK_CHUNK)
        levels += 1
        cur = nchunk * (min(cur, k) if nchunk == 1 else k)
        if nchunk == 1:
            return levels


# (dtype, Nq, Nv, D, n_img)
_CASES = [
    (torch.bfloat16, 77, 256, 512, 300),      # tcgen05 1-CTA, retrieval order, C = 1
    (torch.bfloat16, 77, 256, 128, 1000),     # 1-CTA, retrieval order, C = 5
    (torch.bfloat16, 1, 256, 64, 5000),       # M = 1, retrieval order, C = 10, top-k over two 4096-chunks
    (torch.bfloat16, 250, 1024, 512, 60),     # 2-CTA, 4 sub-tiles, retrieval order, C = 1
    (torch.bfloat16, 77, 1024, 512, 6000),    # cfg 5 flavour (6.3 GB): sub-tiles, retrieval order, two top-k levels
    (torch.bfloat16, 129, 197, 256, 150),     # 2-CTA (M > 128), default order, odd Nv
    (torch.bfloat16, 50, 256, 200, 500),      # SIMT bf16 (D % 64 != 0)
    (torch.float32, 77, 256, 512, 200),       # SIMT fp32
    (torch.bfloat16, 300, 320, 256, 200),     # direction 1: sub-tiles on the query side
    (torch.bfloat16, 77, 256, 512, 100),      # a small gallery: 1-CTA, default order
]
_TEMPS = (1.5, 0.07)


def _case_path(case, direction):
    dtype, Nq, Nv, D, n = case
    if direction == 0:
        return _fwd_path(dtype, Nq, n, Nv, D)
    return _fwd_path(dtype, n * Nv, 1, Nq, D)


def _case_id(case, direction, T):
    dtype, Nq, Nv, D, n = case
    kern, order, C, sub = _case_path(case, direction)
    path = kern + (f"-{order}" if order else "") + (f"-C{C}" if order == "retrieval" else "") + ("-sub" if sub else "")
    lv = _topk_levels(n, min(n, 2048))
    return (f"{'bf16' if dtype == torch.bfloat16 else 'f32'}-{Nq}x{Nv}x{D}-n{n}-dir{direction}-T{T}-{path}"
            + (f"-topk{lv}" if lv > 1 else ""))


_PARAMS = [pytest.param(ci, d, T, id=_case_id(c, d, T)) for ci, c in enumerate(_CASES) for d in (0, 1) for T in _TEMPS]


def test_cases_cover_every_retrieval_path():
    """Together the cases reach every forward path one query against a gallery can take (bar the 'sync' order, which
    needs many query tiles and is the training shapes' order) and multi-level top-k."""
    seen = set()
    for case in _CASES:
        for d in (0, 1):
            kern, order, C, sub = _case_path(case, d)
            seen.add(kern if order is None else f"{kern}-{order}")
            if sub:
                seen.add(f"sub-tiles-dir{d}")
            if order == "retrieval":
                seen.add(f"retrieval-C{'1' if C == 1 else '>1'}")
        if _topk_levels(case[4], min(case[4], 2048)) > 1:
            seen.add("topk-multilevel")
        if case[1] == 1:
            seen.add("M=1")
    want = {"simt-f32", "simt-bf16", "tc1-default", "tc2-default", "tc1-retrieval", "tc2-retrieval",
            "sub-tiles-dir0", "sub-tiles-dir1", "retrieval-C1", "retrieval-C>1", "topk-multilevel", "M=1"}
    assert want <= seen, sorted(want - seen)


# ----------------------------------------------------------------------------------------------------------------
# galleries and their fp64 scores
# ----------------------------------------------------------------------------------------------------------------
def _rel(dtype):
    return 2.0 ** -7 + 2.0 ** -15 if dtype == torch.bfloat16 else 2.0 ** -23


def _reference(q, gal, ids=None, chunk=64):
    """fp64 scores at T = 1 and their tolerance terms, per direction: {d: (score, A, B)} (see the module docstring).
    Scores and tolerances scale with 1/T exactly."""
    q64 = q.double()
    qn = q64.norm(dim=1)
    ids = torch.arange(gal.shape[0], device=gal.device) if ids is None else ids
    out = {0: ([], [], []), 1: ([], [], [])}
    for s in range(0, ids.numel(), chunk):
        g64 = gal[ids[s:s + chunk]].double()                     # (c, Nv, D)
        e = g64 @ q64.T                                          # (c, Nv, Nq): e[n, p, a]
        vn = g64.norm(dim=2)                                     # (c, Nv)
        ae = e.abs()
        out[0][0].append(e.amax(1).mean(1)); out[0][1].append(ae.amax(1).mean(1))
        out[0][2].append(qn.mean() * vn.amax(1))
        out[1][0].append(e.amax(2).mean(1)); out[1][1].append(ae.amax(2).mean(1))
        out[1][2].append(vn.mean(1) * qn.amax())
        del g64, e, ae
    return {d: tuple(torch.cat(x) for x in out[d]) for d in (0, 1)}


def _tolerance(case, direction, T, A, B):
    dtype, Nq, Nv, D, _ = case
    K = Nq if direction == 0 else Nv
    return (_rel(dtype) * A + (1 + 2.0 ** -6) * (D * 2.0 ** -23 * B + (K + 3) * 2.0 ** -24 * A)) / T


def _layout(n, C):
    """Ids of the planted images: the first four get distinct levels, `dups` are (original, copy) pairs.  Copies sit
    a multiple of 32 ids from their original: see _Gallery."""
    C = n if C is None or C >= n else C
    b = C * max(1, (n // 2) // C) if C < n else n // 2           # a C-chunk boundary near the middle
    if n > _TOPK_CHUNK:
        return [0, b - 1, b, _TOPK_CHUNK - 1], [(0, _TOPK_CHUNK), (b, n - 1)]
    step = 32 * max(1, round(n / 128))
    return [0, b - 1, b, n - 1], [(0, step), (n - 1, n - 1 - step)]


class _Gallery:
    def __init__(self, case):
        dtype, Nq, Nv, D, n = case
        dev = torch.device("cuda")
        g = torch.Generator(device=dev).manual_seed(1000 + Nq * 7 + Nv * 13 + D * 17 + n)
        self.q = torch.nn.functional.normalize(torch.randn(Nq, D, device=dev, generator=g), dim=1).to(dtype)
        self.gal = torch.empty(n, Nv, D, dtype=dtype, device=dev)
        for s in range(0, n, 256):
            x = torch.randn(min(256, n - s), Nv, D, device=dev, generator=g)
            self.gal[s:s + x.shape[0]] = torch.nn.functional.normalize(x, dim=2).to(dtype)
            del x
        # the best random image (either direction, in cosine units) bounds the planted levels from below
        ref = _reference(self.q, self.gal)
        ceiling = max(ref[0][0].max().item(), ref[1][0].max().item())
        step = 0.085 if dtype == torch.bfloat16 else 0.02
        levels = [c for c in 0.99 - step * np.arange(32) if c > ceiling + step / 2]
        assert len(levels) >= 4, (ceiling, levels)
        C = _case_path(case, 0)[2]
        first, dups = _layout(n, C)
        # In direction 1 the gallery patches are the forward's rows (image n from row n*Nv) and the mean over them is
        # summed from 32-row partial groups, so two copies add in the same order only when their first rows lie at
        # the same offset within a group.  Where they do not, they may differ in the last bit.
        assert all((b - a) * Nv % 32 == 0 for a, b in dups)
        taken = set(first) | {b for _, b in dups}
        rng = np.random.default_rng(n)
        extra = [int(i) for i in rng.permutation(n) if int(i) not in taken][:len(levels) - len(first)]
        self.distinct = first + extra
        self.dups = dups
        qf = torch.nn.functional.normalize(self.q.float(), dim=1)
        tok = qf[torch.arange(Nv, device=dev) % Nq]                                   # (Nv, D): the token of patch p
        for i, c in zip(self.distinct, levels):
            noise = torch.randn(Nv, D, device=dev, generator=g)
            noise = torch.nn.functional.normalize(noise - (noise * tok).sum(1, keepdim=True) * tok, dim=1)
            self.gal[i] = (c * tok + math.sqrt(1 - c * c) * noise).to(dtype)
        for a, b in dups:
            self.gal[b] = self.gal[a]
        self.planted = sorted(set(self.distinct) | {b for _, b in dups})
        pid = torch.tensor(self.planted, device=dev)
        pref = _reference(self.q, self.gal, pid)
        for d in (0, 1):                                          # patch the planted images into the fp64 scores
            for k in range(3):
                ref[d][k][pid] = pref[d][k]
                for a, b in dups:                                 # the same data: the same score, whatever the GEMM
                    ref[d][k][b] = ref[d][k][a]
        self.ref = ref


_CACHE = {}


@pytest.fixture(scope="module", autouse=True)
def _release_galleries():
    yield
    _CACHE.clear()
    torch.cuda.empty_cache()


def _gallery(ci):
    if ci not in _CACHE:
        _CACHE.clear()                                            # one gallery at a time (the cfg 5 one is 6.3 GB)
        torch.cuda.empty_cache()
        _CACHE[ci] = _Gallery(_CASES[ci])
    return _CACHE[ci]


def _u32(x):
    return np.ascontiguousarray(x, dtype=np.float32).view(np.uint32)


def _checked(ci, direction, T):
    """The kernel's scores, the fp64 scores and tolerances, after checking the planted-score premise."""
    case = _CASES[ci]
    G = _gallery(ci)
    ref0, A, B = G.ref[direction]
    ref = (ref0 / T).cpu().numpy()
    tol = _tolerance(case, direction, T, A, B).cpu().numpy()
    d_ids = np.array(G.distinct)
    lv = np.sort(ref[d_ids])
    gap = np.diff(lv).min()
    assert gap > 10 * tol[G.planted].max(), (gap, tol[G.planted].max())
    rand = np.setdiff1d(np.arange(case[4]), G.planted)
    worst_planted = (ref[G.planted] - tol[G.planted]).min()
    assert worst_planted > (ref[rand] + tol[rand]).max(), "the planted images must outrank every random one"
    got = R._scores(G.q, G.gal, T, direction).cpu().numpy()
    return G, got, ref, tol


@pytest.mark.parametrize("ci,direction,T", _PARAMS)
def test_scores_match_fp64_per_element(ci, direction, T):
    G, got, ref, tol = _checked(ci, direction, T)
    err = np.abs(got.astype(np.float64) - ref)
    bad = np.flatnonzero(~(err <= tol))                           # NaN fails too
    assert bad.size == 0, (f"{bad.size} scores outside their bound, first ids {bad[:8].tolist()}: got "
                           f"{got[bad[:4]].tolist()} want {ref[bad[:4]].tolist()} tol {tol[bad[:4]].tolist()}")
    for a, b in G.dups:
        assert _u32(got[a]) == _u32(got[b]), (a, b, got[a], got[b])


@pytest.mark.parametrize("ci,direction,T", _PARAMS)
def test_retrieve_topk_ranks_like_fp64(ci, direction, T):
    G, got, ref, tol = _checked(ci, direction, T)
    n = got.size
    k = min(n, 2048)
    s, ids = R.retrieve_topk(G.q, G.gal, T, k, direction)
    s, ids = s.cpu().numpy(), ids.cpu().numpy().astype(np.int64)
    # (1) exactly a stable descending sort of the kernel's own scores, scores bit for bit
    assert np.array_equal(ids, np.argsort(-got, kind="stable")[:k])
    assert np.array_equal(_u32(s), _u32(got[ids]))
    # (2) the planted images first, in their fp64 order (the copies right after their lower-id twin)
    P = len(G.planted)
    planted = np.array(G.planted)
    assert np.array_equal(ids[:P], planted[np.argsort(-ref[planted], kind="stable")])
    pos = {int(i): r for r, i in enumerate(ids)}
    for a, b in map(sorted, G.dups):
        assert pos[a] + 1 == pos[b], (a, b, pos[a], pos[b])
    # (3) the rest: every inversion against fp64 is between two scores within tol_a + tol_b
    r, t = ref[ids], tol[ids]
    inv = (r[None, :] - r[:, None]) > (t[None, :] + t[:, None])   # [i, j]: j ranked after i but certainly above it
    assert not np.triu(inv, 1).any(), np.argwhere(np.triu(inv, 1))[:4].tolist()
    if k < n:
        out = np.setdiff1d(np.arange(n), ids)
        assert (ref[out] - tol[out]).max() <= (r + t).min(), "an excluded image certainly outranks an included one"
    if direction == 0 and T == _TEMPS[0]:
        for bad_k in (n + 1, 2049):
            with pytest.raises(TriadError):
                R.retrieve_topk(G.q, G.gal, T, bad_k, direction)


# ----------------------------------------------------------------------------------------------------------------
# C. triad_topk
# ----------------------------------------------------------------------------------------------------------------
def _topk(x: torch.Tensor, k: int):
    lib = _lib.load()
    n = x.numel()
    out_s = torch.empty(k, dtype=torch.float32, device=x.device)
    out_i = torch.empty(k, dtype=torch.int32, device=x.device)
    ws = torch.empty(max(lib.triad_topk_workspace_bytes(n, k), 1), dtype=torch.uint8, device=x.device)
    with ops._on(x):
        check(lib.triad_topk(x.data_ptr(), n, k, out_s.data_ptr(), out_i.data_ptr(), ws.data_ptr(), ws.numel(),
                             ops._stream(x.device)), "triad_topk")
    return out_s.cpu().numpy(), out_i.cpu().numpy().astype(np.int64)


_F32 = np.finfo(np.float32)
_SPECIALS = np.array([np.inf, -np.inf, _F32.max, -_F32.max, _F32.smallest_subnormal, -_F32.smallest_subnormal,
                      _F32.smallest_normal * np.float32(0.5), -_F32.smallest_normal * np.float32(0.5)], np.float32)


def _vector(n, dist, rng):
    if dist == "normal":
        return rng.standard_normal(n).astype(np.float32)
    if dist == "quantised":                                    # 16 levels: ties inside and across every chunk
        return (rng.integers(0, 16, n).astype(np.float32) - 8) / 4
    if dist == "equal":
        return np.full(n, 0.75, np.float32)
    if dist == "ascending":
        return np.arange(n, dtype=np.float32)
    assert dist == "specials"
    if n <= 2:
        return np.array([-0.0, 0.0], np.float32)[:n]           # a -0.0 before a +0.0: the lower id goes first
    # negative numbers, a few of each special value, and +-0 in between: the top 100 crosses the zeros
    x = -np.abs(rng.standard_normal(n)).astype(np.float32)
    pos = rng.permutation(n)
    m = min(8, n // 24)
    for s, v in enumerate(_SPECIALS):
        x[pos[s * m:(s + 1) * m]] = v
    nz = min(40, (n - 8 * m) // 2)
    x[pos[8 * m:8 * m + nz]] = np.float32(0.0)
    x[pos[8 * m + nz:8 * m + 2 * nz]] = np.float32(-0.0)
    return x


_TOPK_N = [1, 2, 4095, 4096, 4097, 12289, 100_000, (1 << 22) + 3]
_TOPK_DISTS = ["normal", "quantised", "equal", "ascending", "specials"]


@pytest.mark.parametrize("dist", _TOPK_DISTS)
@pytest.mark.parametrize("n", _TOPK_N)
def test_topk_is_a_stable_descending_argsort(n, dist):
    rng = np.random.default_rng(n * 10 + _TOPK_DISTS.index(dist))
    x = _vector(n, dist, rng)
    order = np.argsort(-x, kind="stable")
    xd = torch.from_numpy(x).cuda()
    ks = sorted({k for k in (1, 10, 100, 2047, 2048) if k <= n} | ({n} if n <= 2048 else set()))
    for k in ks:
        s, ids = _topk(xd, k)
        assert np.array_equal(ids, order[:k]), (k, np.flatnonzero(ids != order[:k])[:8].tolist())
        assert np.array_equal(_u32(s), _u32(x[order[:k]])), k
    if dist == "specials" and n >= 100:                          # the top 100 reaches zeros of both signs
        z = x[order[:100]]
        z = z[z == 0]
        assert np.signbit(z).any() and not np.signbit(z).all()


# ----------------------------------------------------------------------------------------------------------------
# D. triad_diag_ranks, compute_recall_at_k
# ----------------------------------------------------------------------------------------------------------------
def _diag_ranks(sim: torch.Tensor):
    lib = _lib.load()
    N = sim.shape[0]
    ranks = torch.empty(N, dtype=torch.int32, device=sim.device)
    with ops._on(sim):
        check(lib.triad_diag_ranks(sim.data_ptr(), N, ranks.data_ptr(), ops._stream(sim.device)), "triad_diag_ranks")
    return ranks.cpu().numpy()


def _matrix(N, kind, rng):
    if kind == "all_nan":
        return np.full((N, N), np.nan, np.float32)
    if kind == "quantised":                                      # 6 levels: the diagonal ties earlier and later columns
        sim = rng.integers(0, 6, (N, N)).astype(np.float32) / 2
    else:
        sim = rng.standard_normal((N, N)).astype(np.float32)
        sim[np.diag_indices(N)] += np.float32(2.0)               # recall well inside (0, 1)
    diag = np.diag_indices(N)
    if kind == "ties":                                           # the diagonal copied to a column on each side
        for i in range(N):
            for j in (i - 1 - i % 3, i + 1 + i % 5):
                if 0 <= j < N:
                    sim[i, j] = sim[i, i]
    elif kind == "inf_zero":
        mask = rng.random((N, N)) < 0.2
        sim[mask] = rng.choice(np.array([np.inf, -np.inf, 0.0, -0.0], np.float32), mask.sum())
        sim[diag] = rng.choice(np.array([np.inf, -np.inf, 0.0, -0.0, 1.0], np.float32), N)
    elif kind == "nan_off":
        mask = rng.random((N, N)) < 0.1
        mask[diag] = False
        sim[mask] = np.nan
    elif kind == "nan_diag":
        sim[rng.random((N, N)) < 0.1] = np.nan
        sim[diag[0][::2], diag[1][::2]] = np.nan                 # every other row: NaN diagonal
    return sim


def _ref_ranks(sim):
    return np.array([int(np.flatnonzero(np.argsort(-sim[i], kind="stable") == i)[0]) for i in range(sim.shape[0])])


_RANK_KINDS = ["normal", "quantised", "ties", "inf_zero", "nan_off", "nan_diag", "all_nan"]


@pytest.mark.parametrize("kind", _RANK_KINDS)
@pytest.mark.parametrize("N", [1, 31, 255, 256, 257, 1000, 3001])
def test_diag_ranks_and_recall_match_a_stable_argsort(N, kind):
    sim = _matrix(N, kind, np.random.default_rng(N * 10 + _RANK_KINDS.index(kind)))
    want = _ref_ranks(sim)
    got = _diag_ranks(torch.from_numpy(sim).cuda())
    bad = np.flatnonzero(got != want)
    assert bad.size == 0, [(int(i), int(got[i]), int(want[i]), float(sim[i, i])) for i in bad[:6]]
    rec = R.compute_recall_at_k(sim)
    assert rec == {f"r{k}": float(np.mean(want < k)) for k in (1, 5, 10, 20)}
    if kind in ("all_nan", "nan_diag") and N > 1:
        assert rec["r1"] < 1.0                                   # NaN scores never read as perfect recall


# ----------------------------------------------------------------------------------------------------------------
# E. triad_similarity_matrix
# ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("T", [1.5, 0.07])
@pytest.mark.parametrize("B,N1,N2,D", [(1, 1, 1, 8), (2, 9, 65, 33), (3, 17, 130, 512), (1, 8, 64, 1000)])
def test_similarity_matrix_matches_fp64(B, N1, N2, D, T):
    lib = _lib.load()
    g = torch.Generator().manual_seed(B * 1000 + N1 * 100 + N2 + D)
    f1 = torch.randn(B, N1, D, generator=g) * 3
    f2 = torch.randn(B, N2, D, generator=g) * 0.01
    f1[0, -1] = 0                                                # zero rows: F.normalize's eps keeps them at 0
    f2[-1, 0] = 0
    out = torch.full((B, N1, N2), float("nan"), device="cuda")
    f1d, f2d, Td = f1.cuda(), f2.cuda(), torch.tensor(T, device="cuda")
    with ops._on(out):
        check(lib.triad_similarity_matrix(f1d.data_ptr(), f2d.data_ptr(), Td.data_ptr(), B, N1, N2, D,
                                          out.data_ptr(), ops._stream(out.device)), "triad_similarity_matrix")
    n1 = f1.double() / f1.double().norm(dim=2, keepdim=True).clamp(min=1e-12)
    n2 = f2.double() / f2.double().norm(dim=2, keepdim=True).clamp(min=1e-12)
    want = torch.bmm(n1, n2.transpose(1, 2)) * float(np.float32(T))
    err = (out.cpu().double() - want).abs()
    assert bool((err <= 1e-5 * T).all()), (err.max().item(), torch.nonzero(~(err <= 1e-5 * T))[:4].tolist())
    assert bool((out[0, -1] == 0).all()) and bool((out[-1, :, 0] == 0).all())
