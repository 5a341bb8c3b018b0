"""GPU tier: retrieval over a ragged caption gallery (``RaggedGallery``, ``triad_retrieve_scores_ragged``).

A. An exact probe: small-integer operands, T = 1/2 and power-of-two token counts, so every product, bf16 rounding,
   weight and fp32 sum is exact and each caption's maximum sits at a known token.  Both directions must equal fp64
   bit for bit; this pins the caption boundaries inside the 256-row slots, the zero rows after a slot's last caption
   (they must not join a maximum) and the 1/length weights of direction 1.
B. Scores of random unit-norm galleries against fp64 of the stored bf16 operands, per caption, with the tolerance
   of tests/test_gpu_retrieval.py restated: with e = <q_a, v_t> / T in fp64,
       tol_c = (rel A_c + (1 + 2^-6) (D 2^-23 B_c + (K + 3) 2^-24 A_c)) / T,   rel = 2^-7 + 2^-15,
   A_c = mean max |e| and B_c = mean max |q_a| |v_t| in the score's own order, K = the number of terms of the mean
   (the query's Nq in direction 0, the caption's length in direction 1, where its rows are summed one by one).
   The cases sweep Nq in {1, 77, 129, 256, 1024}, slot counts on both sides of the forward's 48 MB / 16 MB tile-order
   thresholds, cfg 3's caption lengths U[8, 77] and galleries of 1-token and 256-token captions, at T = 1.5 and 0.07;
   a test asserts that together they reach each forward path they were written for.
C. The reference's aggregator_tv_v2t / aggregator_tv_t2v per caption, and pairwise_similarity's row for one image.
D. Zero padding is not equivalent: a gallery whose zero-padded form ranks differently, in both directions.
E. Repeated calls are bit-identical, a caption's score does not depend on the captions packed before it, and a
   query makes no host synchronisation.
F. Gallery-sharded top-k: one rank against retrieve_topk; two ranks under NCCL (skipped on one GPU).
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from triad_b200 import retrieval as R

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = torch.device("cuda")
_SMS = torch.cuda.get_device_properties(0).multi_processor_count if torch.cuda.is_available() else 148
_MiB = 1 << 20
SLOT = 256


def _captions(lengths, D, seed, scale=None):
    """A list of unit-norm bf16 captions [L_i, D] (or small-integer ones when scale is given)."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    total = int(np.sum(lengths))
    if scale is None:
        flat = torch.nn.functional.normalize(torch.randn(total, D, generator=g, device=DEV), dim=1).bfloat16()
    else:
        flat = torch.randint(-scale, scale + 1, (total, D), generator=g, device=DEV).bfloat16()
    return list(torch.split(flat, [int(x) for x in lengths]))


def _segments(gal: R.RaggedGallery):
    """Caption id of every slot row (n_cap for the zero rows at a slot's end)."""
    info = gal.cap_info.cpu().numpy()
    cid = np.full(gal.n_slots * SLOT, len(gal), dtype=np.int64)
    for c, (r, n) in enumerate(info):
        cid[r:r + n] = c
    return torch.from_numpy(cid).to(DEV)


def _fp64(q, gal: R.RaggedGallery, direction):
    """fp64 scores at T = 1 and the tolerance terms (A, B, K) per caption, from the stored bf16 rows."""
    n = len(gal)
    cid = _segments(gal)
    keep = cid < n
    rows = gal.slots[keep].double()
    cid = cid[keep]
    q64 = q.double()
    e = rows @ q64.T                                             # [rows, Nq]
    qn, vn = q64.norm(dim=1), rows.norm(dim=1)
    lens = torch.from_numpy(gal.lengths.astype(np.int64)).to(DEV)
    if direction == 0:
        def segmax(x):
            out = torch.full((n, x.shape[1]), -float("inf"), dtype=torch.float64, device=DEV)
            return out.scatter_reduce_(0, cid[:, None].expand_as(x), x, "amax", include_self=True)
        s = segmax(e).mean(1)
        A = segmax(e.abs()).mean(1)
        B = qn.mean() * torch.zeros(n, dtype=torch.float64, device=DEV).scatter_reduce_(0, cid, vn, "amax")
        K = torch.full((n,), q.shape[0], dtype=torch.float64, device=DEV)
    else:
        def segmean(x):
            return torch.zeros(n, dtype=torch.float64, device=DEV).index_add_(0, cid, x) / lens
        s = segmean(e.amax(1))
        A = segmean(e.abs().amax(1))
        B = segmean(vn) * qn.amax()
        K = lens.double()
    return s, A, B, K


def _tolerance(D, T, A, B, K):
    rel = 2.0 ** -7 + 2.0 ** -15
    return (rel * A + (1 + 2.0 ** -6) * (D * 2.0 ** -23 * B + (K + 3) * 2.0 ** -24 * A)) / T


# ----------------------------------------------------------------------------------------------------------------
# which forward path a call takes (launch_maxmean_tc's tile order, restated)
# ----------------------------------------------------------------------------------------------------------------
def _path(Nq, n_slots, D, direction, sms=_SMS):
    if direction == 1:                                           # rows = slot rows: cta_group::2, one image
        return "tc2", "default", 1, Nq > 256
    cta = 1 if Nq <= 128 else 2
    n_m = -(-Nq // (128 * cta))
    img = SLOT * D * 2
    clusters = sms // cta
    order, C = "default", n_slots
    if n_slots * img > 48 * _MiB:
        c16 = max(1, 16 * _MiB // img)
        if n_m * c16 >= 4 * clusters:
            order, C = "sync", min(c16, n_slots)
        else:
            order, C = "retrieval", min(max(1, min(64, 48 * _MiB // (clusters * img))), n_slots)
    return f"tc{cta}", order, C, False


def _lengths(spec, n, seed):
    if spec == "cfg3":
        return np.random.default_rng(seed).integers(8, 78, size=n)
    return np.full(n, int(spec))


# (Nq, D, lengths, captions, path the direction-0 call is written for)
_CASES = [
    (77, 512, "cfg3", 600, "tc1-default"),             # ~100 slots, 26 MB: below the 48 MB threshold
    (77, 512, "cfg3", 2000, "tc1-retrieval-C1"),       # ~340 slots, 86 MB
    (1, 128, "cfg3", 6000, "tc1-retrieval-C>1"),       # one query token, ~1000 slots of 64 KB
    (129, 256, "1", 12800, "tc2-default"),             # 1-token captions: 256 per slot, 50 slots
    (256, 512, "256", 300, "tc2-retrieval-C>1"),       # 256-token captions: one per slot, 79 MB
    (1024, 256, "cfg3", 2500, "tc2-sync"),             # ~420 slots of 128 KB with four query tiles
    (1024, 512, "cfg3", 800, "tc2-default"),           # direction 1: four 256-token sub-tiles of the query
]
_TEMPS = (1.5, 0.07)


def _label(kern, order, C, sub):
    return kern + "-" + order + (("-C1" if C == 1 else "-C>1") if order == "retrieval" else "") + ("-sub" if sub else "")


_GAL = {}


def _case(ci):
    if ci not in _GAL:
        _GAL.clear()
        Nq, D, spec, n, _ = _CASES[ci]
        lens = _lengths(spec, n, 100 + ci)
        gal = R.RaggedGallery.from_list(_captions(lens, D, 200 + ci))
        g = torch.Generator(device=DEV).manual_seed(300 + ci)
        q = torch.nn.functional.normalize(torch.randn(Nq, D, generator=g, device=DEV), dim=1).bfloat16()
        _GAL[ci] = (q, gal, {d: _fp64(q, gal, d) for d in (0, 1)})
    return _GAL[ci]


@pytest.fixture(scope="module", autouse=True)
def _release():
    yield
    _GAL.clear()
    torch.cuda.empty_cache()


def test_cases_reach_the_paths_they_were_written_for():
    seen = set()
    for ci, (Nq, D, spec, n, want) in enumerate(_CASES):
        n_slots = R.ragged_plan(_lengths(spec, n, 100 + ci))[0].shape[0]
        assert _label(*_path(Nq, n_slots, D, 0)) == want, (ci, _path(Nq, n_slots, D, 0))
        seen.add(want)
        seen.add(_label(*_path(Nq, n_slots, D, 1)))
    assert {"tc1-default", "tc2-default", "tc1-retrieval-C1", "tc1-retrieval-C>1", "tc2-retrieval-C>1", "tc2-sync",
            "tc2-default-sub"} <= seen, seen
    assert {c[0] for c in _CASES} >= {1, 77, 129, 256, 1024}


# ----------------------------------------------------------------------------------------------------------------
# A. exact probe
# ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("Nq", [4, 512])
def test_exact_probe_both_directions(Nq):
    D = 64
    pattern = [1, 2, 64, 4, 128, 32, 8, 16, 256, 1, 1, 32, 64, 128, 2, 4, 8, 16, 32, 1, 256, 2]
    lens = np.array(pattern * 3)
    caps = _captions(lens, D, 11, scale=2)
    # one caption's maximum over its tokens is planted at its last token for query token 0: (all ones) . q_0 > any
    q = torch.randint(-1, 2, (Nq, D), generator=torch.Generator(device=DEV).manual_seed(12), device=DEV).bfloat16()
    q[0] = 1
    caps[5][-1] = 2
    gal = R.RaggedGallery.from_list(caps)
    assert gal.n_slots > 3
    T = 0.5
    for d in (0, 1):
        s64 = _fp64(q, gal, d)[0] / T
        got = R._scores_ragged(q, gal, T, d).double()
        assert torch.equal(got, s64), (d, (got - s64).abs().max().item())
    # the planted maximum: query token 0 meets 128 at caption 5's last token, which no gap row or neighbour can hide
    e = (caps[5].double() @ q.double().T)
    assert e[-1, 0] == 128 and e[:-1, 0].max() < 128


# ----------------------------------------------------------------------------------------------------------------
# B. scores against fp64
# ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ci", range(len(_CASES)))
@pytest.mark.parametrize("direction", [0, 1])
@pytest.mark.parametrize("T", _TEMPS)
def test_scores_match_fp64(ci, direction, T):
    q, gal, ref = _case(ci)
    s, A, B, K = ref[direction]
    D = gal.shape[1]
    tol = _tolerance(D, T, A, B, K)
    got = R._scores_ragged(q, gal, T, direction).double()
    err = (got - s / T).abs()
    worst = (err / tol).max().item()
    print(f"ragged case {ci} dir {direction} T {T}: n_cap {len(gal)} slots {gal.n_slots} worst err/tol {worst:.3f}")
    assert torch.isfinite(got).all()
    assert (err <= tol).all(), worst
    # top-k is the kernel's own scores' stable descending order
    k = min(10, len(gal))
    ts, ti = R.retrieve_topk(q, gal, T, k, direction)
    order = torch.from_numpy(np.argsort(-got.cpu().numpy(), kind="stable")[:k]).to(DEV)
    assert torch.equal(ti.long(), order) and torch.equal(ts.double(), got[order])


# ----------------------------------------------------------------------------------------------------------------
# C. the reference and pairwise_similarity
# ----------------------------------------------------------------------------------------------------------------
@pytest.fixture()
def ref_retrieval():
    from oracle import ref_loader
    ref = ref_loader.load()
    if ref is None:
        pytest.skip("oracle/_ref not staged")
    return ref[1]


def test_matches_the_reference_aggregators(ref_retrieval):
    D, T = 128, 0.07
    lens = _lengths("cfg3", 300, 21)
    caps = _captions(lens, D, 22)
    image = torch.nn.functional.normalize(torch.randn(49, D, generator=torch.Generator(device=DEV).manual_seed(23),
                                                      device=DEV), dim=1).bfloat16()
    gal = R.RaggedGallery.from_list(caps)
    got = {d: R._scores_ragged(image, gal, T, d).double() for d in (0, 1)}
    for d in (0, 1):
        _, A, B, K = _fp64(image, gal, d)
        tol = _tolerance(D, T, A, B, K) + 2.0 ** -20 * A / T          # + the reference's own fp32 rounding
        agg = ref_retrieval.aggregator_tv_v2t if d == 0 else ref_retrieval.aggregator_tv_t2v
        want = torch.tensor([agg(c.float(), image.float(), T) for c in caps], dtype=torch.float64, device=DEV)
        assert ((got[d] - want).abs() <= tol).all(), d


def test_row_of_pairwise_similarity():
    D, T = 128, 1.5
    lens = _lengths("cfg3", 200, 31)
    caps = _captions(lens, D, 32)
    image = torch.nn.functional.normalize(torch.randn(64, D, generator=torch.Generator(device=DEV).manual_seed(33),
                                                      device=DEV), dim=1).bfloat16()
    gal = R.RaggedGallery.from_list(caps)
    # direction 0 sums the same 32-row groups of the image's tokens in the same order as the dense forward: bit-equal
    row0 = R.pairwise_similarity([image], caps, T, 0)[0]
    assert torch.equal(R._scores_ragged(image, gal, T, 0), row0)
    # direction 1 adds a caption's rows in token order, the dense forward in 32-row groups of the stacked captions
    row1 = R.pairwise_similarity([image], caps, T, 1)[0].double()
    _, A, B, K = _fp64(image, gal, 1)
    assert ((R._scores_ragged(image, gal, T, 1).double() - row1).abs() <= 2 * _tolerance(D, T, A, B, K)).all()


def test_from_padded_keeps_the_masked_rows():
    D = 64
    g = torch.Generator(device=DEV).manual_seed(41)
    feats = torch.randn(5, 77, D, generator=g, device=DEV)                 # fp32: rounded to bf16 at build time
    lens = [77, 1, 30, 8, 64]
    mask = torch.zeros(5, 77, dtype=torch.int64)
    for i, n in enumerate(lens):
        mask[i, :n] = 1
    mask[3, 40] = 1                                                        # a hole-y mask keeps its rows in order
    gal = R.RaggedGallery.from_padded(feats, mask)
    ref = R.RaggedGallery.from_list([feats[i][mask[i].bool().to(DEV)].bfloat16() for i in range(5)])
    assert gal.lengths.tolist() == [77, 1, 30, 9, 64]
    assert torch.equal(gal.slots, ref.slots) and torch.equal(gal.meta, ref.meta) and torch.equal(gal.cap_info, ref.cap_info)
    info = gal.cap_info.cpu().numpy()
    assert torch.equal(gal.slots[info[2, 0]:info[2, 0] + 30], feats[2, :30].bfloat16())
    with pytest.raises(ValueError):
        R.RaggedGallery.from_padded(feats, torch.zeros(5, 77, dtype=torch.int64))


# ----------------------------------------------------------------------------------------------------------------
# D. zero padding is not equivalent
# ----------------------------------------------------------------------------------------------------------------
def test_padding_is_not_equivalent(ref_retrieval):
    D, T, Nq = 64, 1.0, 4
    image = torch.zeros(Nq, D, device=DEV, dtype=torch.bfloat16)
    image[:, 0] = 1
    lens = [3, 5, 2, 2, 70, 40]
    # token t of caption c has <image token, token> = level[c][t]: direction 0 scores max level, direction 1 its mean
    levels = [[-3, -1, -2], [-6, -4, -5, -7, -4], [-0.5, -2], [10, 10], [5] * 70, [2] * 40]
    caps = []
    for lv in levels:
        c = torch.zeros(len(lv), D, device=DEV)
        c[:, 0] = torch.tensor(lv, device=DEV)
        caps.append(c.bfloat16())
    gal = R.RaggedGallery.from_list(caps)
    padded = torch.zeros(len(caps), 77, D, device=DEV, dtype=torch.bfloat16)
    for i, c in enumerate(caps):
        padded[i, :c.shape[0]] = c
    k = len(caps)
    for d, agg in ((0, ref_retrieval.aggregator_tv_v2t), (1, ref_retrieval.aggregator_tv_t2v)):
        want = np.array([agg(c.float(), image.float(), T) for c in caps])
        want_ids = np.argsort(-want, kind="stable")
        _, ids = R.retrieve_topk(image, gal, T, k, d)
        _, pids = R.retrieve_topk(image, padded, T, k, d)
        assert ids.cpu().numpy().tolist() == want_ids.tolist(), d
        assert pids.cpu().numpy().tolist() != want_ids.tolist(), d
    # direction 0 under padding: every all-negative caption scores 0; direction 1 divides by 77
    assert (R._scores(image, padded, T, 0)[:3] == 0).all()
    assert R._scores(image, padded, T, 1)[3].item() == pytest.approx(20 / 77, rel=1e-2)


# ----------------------------------------------------------------------------------------------------------------
# E. determinism, position independence, no host synchronisation
# ----------------------------------------------------------------------------------------------------------------
def test_deterministic_and_position_independent():
    D, Nq = 256, 300
    lens = _lengths("cfg3", 500, 51)
    caps = _captions(lens, D, 52)
    q = torch.nn.functional.normalize(torch.randn(Nq, D, generator=torch.Generator(device=DEV).manual_seed(53),
                                                  device=DEV), dim=1).bfloat16()
    gal = R.RaggedGallery.from_list(caps)
    for prefix in (np.array([1]), np.array([17, 200]), _lengths("cfg3", 37, 54)):
        pre = _captions(prefix, D, 55)
        shifted = R.RaggedGallery.from_list(pre + caps)
        joined = R.RaggedGallery.cat([R.RaggedGallery.from_list(pre), gal])
        for d in (0, 1):
            s = R._scores_ragged(q, gal, 0.07, d)
            assert torch.equal(R._scores_ragged(q, gal, 0.07, d), s)
            assert torch.equal(R._scores_ragged(q, shifted, 0.07, d)[len(pre):], s), (d, prefix.tolist())
            assert torch.equal(R._scores_ragged(q, joined, 0.07, d)[len(pre):], s), (d, prefix.tolist())


def test_no_host_synchronisation():
    D = 512
    gal = R.RaggedGallery.from_list(_captions(_lengths("cfg3", 3000, 61), D, 62))
    q = torch.randn(256, D, device=DEV).bfloat16()
    T = torch.tensor(0.07, device=DEV)
    ref = {d: R.retrieve_topk(q, gal, T, 10, d) for d in (0, 1)}          # workspaces allocated
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        out = {d: R.retrieve_topk(q, gal, T, 10, d) for d in (0, 1)}
    finally:
        torch.cuda.set_sync_debug_mode("default")
    for d in (0, 1):
        assert torch.equal(out[d][1], ref[d][1]) and torch.equal(out[d][0], ref[d][0])


# ----------------------------------------------------------------------------------------------------------------
# F. gallery-sharded top-k
# ----------------------------------------------------------------------------------------------------------------
def test_sharded_single_rank_matches_retrieve_topk():
    from triad_b200.dist import sharded_retrieve_topk
    D = 128
    lens = _lengths("cfg3", 700, 71)
    caps = _captions(lens, D, 72)
    caps[650] = caps[17]                                                   # a tie
    q = torch.nn.functional.normalize(torch.randn(77, D, device=DEV), dim=1).bfloat16()
    gal = R.RaggedGallery.from_list(caps)
    for d in (0, 1):
        s, ids = sharded_retrieve_topk(q, gal, 1.5, 12, 0, direction=d)
        s0, i0 = R.retrieve_topk(q, gal, 1.5, 12, d)
        assert torch.equal(ids, i0.long()) and torch.equal(s, s0)
        # a shard built from its own caption range scores exactly those captions of the whole gallery
        shard = R.RaggedGallery.from_list(caps[300:])
        assert torch.equal(R._scores_ragged(q, shard, 1.5, d), R._scores_ragged(q, gal, 1.5, d)[300:])
        s1, i1 = sharded_retrieve_topk(q, shard, 1.5, 12, 300, direction=d)
        assert (i1 >= 300).all()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs at least 2 GPUs")
def test_sharded_ragged_retrieval_under_nccl():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr", "127.0.0.1", "--master-port", "29521", os.path.join("tools", "sharded_retrieval_check.py"),
           "--ragged"]
    r = subprocess.run(cmd, cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    assert "SHARDED_RETRIEVAL_OK" in r.stdout
