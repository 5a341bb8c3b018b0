"""The projection head (``triad_project_tokens`` forward, ``triad_project_tokens_bwd`` backward with the head products of
``launch_head_gemm``) against an fp64 evaluation of the autocast recipe, per row, per element and per gradient block,
at the LayerNorm's and the L2 normalisation's edges and at the token counts training runs.

Reference.  ``tests.helpers.head_fp64`` on the device: bf16 x, W1 and W2, a = x . W1^T + bf16(b1), h = bf16(a), the
LayerNorm in fp64 (y), ln = bf16(y), out = ln . W2^T + bf16(b2); the gradients are fp64 autograd of the same graph
(the roundings pass gradients straight through).  With ``normalize=True`` the reference is o / max(||o||, 1e-12) in
fp64 of o = bf16(out), the rounding of o resolved as the kernel resolved it: o is the kernel's own ``normalize=False``
output (the same accumulator, bit for bit), which the first check has pinned to bf16(out).

Rounding model, and the bounds it gives.  u(v) is one bf16 ulp of v; bf16(v - e) != bf16(v + e) marks a value within e
of a rounding midpoint ("near-midpoint": the kernel may round it either way).

* fp32 products on the tensor core: |acc - exact| <= 2^-20 sqrt(K) ||p||_2 over the K products p of an element.  This
  is above the 4 sigma random walk of round-to-nearest adds and above K/16 directed roundings of one ulp each on partial
  sums up to 2 ||p||_2, for every K <= 2048 used here.
* The LayerNorm in fp32: the two-pass variance adds 512 squares in order, 4 sigma of the random walk of their
  round-to-nearest errors is below 2^-18 of the sum; rsqrtf (2 ulp) and the affine add a few 2^-24.  So
  |y32 - y64| <= 2^-18 |x^ g| + 2^-22 (|x^ g| + |beta|) when the row sum of h is exact in fp32 (checked per row: h on a
  common power-of-two grid, sum and spread within 24 bits of it), plus 2^-18 mean|h| rstd |g| where it is not.  A one-ulp change of h_k (see below) moves mean and rstd: + 2 |g| (1 + |x^|) rstd / 512 *
  sum_k u(h_k) (1 + |x^_k|) over the row's near-midpoint h.
* Exact-GEMM-1 cases: x small integers (or powers of two) and W1 in {0, +-2^-6}, b1 on a 2^-7 grid, so the first
  product and a are exact in any fp32 order and h is bit-identical to the reference's.  Each output element must be
  bf16(out) or, where out lies within e_o of a midpoint, its neighbour:
      e_o = 2^-20 sqrt(512) ||ln_k W2_jk||_2 + 2^-23 |out| + sum_k [ln_k near-midpoint] u(ln_k) |W2_jk|.
  The near-midpoint count is reported and must stay below a quarter of the elements, or 8 (one near-midpoint ln_k widens
  every output of its row by u(ln_k) |W2_jk|, about 2^-12.5 of |out_j|).
* Random cases (Gaussian x and weights, non-trivial b1, gamma, beta, b2): h may flip where a lies within the first
  product's bound of a midpoint (K = Din); each such flip adds u(h_k) rstd |g_k| to ln_k's deviation.  Per row,
      ||got - out||_2 <= 2^-9 ||out||_2 + (1 + 2^-9) ||e_o||_2      (2^-9: the output rounding),
  with e_o as above and the flipped h counted among the near-midpoint ln.  Every row passes on its own.
* ``normalize=True``: the kernel sums Dout squares in fp32 and takes sqrtf, a division and a product: within
  (Dout + 8) 2^-24 relative before the output rounding; every element is checked as above.
* Gradients, per block against fp64 (dx per 128-row tile x 256 columns, dW1 and dW2 per 128 x 128, the vectors per 64
  elements), each relative to its block's reference norm with a floor of 1e-3 of the whole gradient's norm:
  dx = bf16(bf16(gh) . W1) and dW1 = bf16(gh)^T . x round twice / once at 2^-9: 2^-8; dW2 (bf16 ln, as the reference),
  d gamma, d beta and d b1 (fp32 sums of fp32 terms, rare one-ulp h / ln flips): 2^-10; d b2 sums bf16 gy in fp32:
  2^-14.  And, as in tests/test_gpu_projection_backward.py, no gradient is further from fp64 (Frobenius) than the
  torch closed form the kernels replaced.

Routes.  The forward has one kernel; a case reports its tiles, the last tile's rows, k-blocks and the column halves.
The backward's three products take the split plan of ``plan_head_splits`` (dense_gemm.cu), restated in ``_plan``; the
restatement is pinned to the library through ``triad_project_tokens_bwd_workspace_bytes`` (CPU tier), and
``test_every_regime_has_a_case`` asserts that the cases cover every regime of ``REGIMES``.

Every run prints one JSON line (pytest -s): the route, how close each check came to its bound, the near-midpoint
counts, the LayerNorm edge statistics and the peak device memory.
"""
import json
import math
from dataclasses import dataclass

import pytest
import torch

from tests.helpers import head_fp64

HIDDEN = 512
ACC = 2.0 ** -20                 # fp32 tensor-core accumulation: 2^-20 sqrt(K) ||p||_2
LN_SUM, LN_OP = 2.0 ** -18, 2.0 ** -22
GRAD_TOL = {"dx": 2.0 ** -8, "dw1": 2.0 ** -8, "db1": 2.0 ** -10, "dg": 2.0 ** -10, "db": 2.0 ** -10,
            "dw2": 2.0 ** -10, "db2": 2.0 ** -14}
BLOCKS = {"dx": (128, 256), "dw1": (128, 128), "db1": (1, 64), "dg": (1, 64), "db": (1, 64), "dw2": (128, 128),
          "db2": (1, 64)}
NAMES = ("dx", "dw1", "db1", "dg", "db", "dw2", "db2")
# against the closed form: err(kernels) <= SLACK * err(closed form) + ABS_SLACK (tests/test_gpu_projection_backward.py)
SLACK, ABS_SLACK = 1.25, 2e-5

#: regimes of the backward's head products, and what puts a case in one (``_plan``)
REGIMES = {
    "weight_multi_kblock_short_last": "dW1 or dW2 items of more than one k-block, the last split shorter than the others",
    "dx_pick_splits": "dx with at least as many (row tile, slice) units as CTA pairs: the shared pick_splits heuristic",
    "slices_and_multi_kblock": "more than one 512-column slice together with more than one k-block per item",
    "finish_over_16_tiles": "proj_bwd_finish_kernel adds more than 16 tile partials",
}


@dataclass
class Case:
    name: str
    M: int
    Din: int
    Dout: int
    exact: bool                  # exact-GEMM-1 inputs (see the module docstring) or Gaussian
    edge: str = ""               # "small_var" | "large_mean" | "l2_zero": LayerNorm / L2 edge rows, in exact cases
    eps: float = 1e-5
    fwd: bool = True
    bwd: bool = False
    seed: int = 0


CASES = [
    Case("e_m1_d64_o16", 1, 64, 16, True, seed=1),
    Case("r_m127_d576_o48", 127, 576, 48, False, seed=2),
    Case("e_m128_d2048_o272", 128, 2048, 272, True, seed=3),
    Case("r_m129_d1536_o496", 129, 1536, 496, False, seed=4),
    Case("e_m256_d768_o256", 256, 768, 256, True, seed=5),
    Case("r_m257_d64_o512", 257, 64, 512, False, seed=6),
    Case("e_m257_d576_o496", 257, 576, 496, True, seed=7),
    # LayerNorm edges (forward and backward) and the L2 normalisation's zero row
    Case("e_smallvar_eps1e-5", 257, 576, 272, True, "small_var", 1e-5, bwd=True, seed=8),
    Case("e_smallvar_eps1e-3", 129, 768, 512, True, "small_var", 1e-3, bwd=True, seed=9),
    Case("e_largemean", 256, 64, 48, True, "large_mean", bwd=True, seed=10),
    Case("e_l2zero", 127, 2048, 16, True, "l2_zero", seed=11),
    # a split shorter than the others in all three products, 21 tile partials
    Case("r_bwd_m2600_d576_o272", 2600, 576, 272, False, fwd=False, bwd=True, seed=12),
    # training token counts: audio 256 x 250, visual 256 x 256, text 512 x 77, a 1536-wide encoder
    Case("r_audio_256x250_d768", 64000, 768, 512, False, bwd=True, seed=13),
    Case("e_audio_256x250_d768", 64000, 768, 512, True, seed=14),
    Case("r_visual_256x256_d768", 65536, 768, 512, False, bwd=True, seed=15),
    Case("r_text_512x77_d768", 39424, 768, 512, False, bwd=True, seed=16),
    Case("r_256x256_d1536", 65536, 1536, 512, False, bwd=True, seed=17),
]
BWD_CASES = [c for c in CASES if c.bwd]


# ---- the split plan of the head products (dense_gemm.cu plan_head_splits / pick_splits), restated -------------------
def _cdiv(a, b):
    return -(-a // b)


def _pick_splits(n_tiles, nkb, n_clusters):
    best, best_eff = 1, 0.0
    for s in (1, 2, 3, 4, 6, 8, 12, 16):
        if s > nkb:
            break
        items = n_tiles * s
        eff = items / (_cdiv(items, n_clusters) * n_clusters) - 0.01 * (s - 1)
        if eff > best_eff + 1e-9:
            best_eff, best = eff, s
    return best


def _plan(M, Kc, D, mode, sms):
    clusters = sms // 2
    rows, K = (M, Kc) if mode == 0 else (Kc, M)
    n_tiles, n_slices, nkb = _cdiv(rows, 256), _cdiv(D, 512), _cdiv(K, 64)
    units = n_tiles * n_slices
    branch = "pick_splits" if units >= clusters else "fill"
    splits = _pick_splits(units, nkb, clusters) if units >= clusters else clusters // units
    kbs = _cdiv(nkb, max(1, min(splits, nkb)))
    splits = _cdiv(nkb, kbs)
    return {"branch": branch, "rows": rows, "D": D, "slices": n_slices, "k_blocks": nkb, "splits": splits,
            "kb_per_split": kbs, "last_split_kb": nkb - (splits - 1) * kbs}


def _bwd_plans(M, Din, Dout, sms):
    return {"dw2": _plan(M, Dout, HIDDEN, 1, sms),     # gy^T . ln
            "dw1": _plan(M, HIDDEN, Din, 1, sms),      # gh^T . x
            "dx": _plan(M, HIDDEN, Din, 0, sms)}       # gh . W1


def _sms():
    if torch.cuda.is_available():
        return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    return 148                                         # what the library assumes without a device


def _regimes(M, Din, Dout, sms):
    p = _bwd_plans(M, Din, Dout, sms)
    out = set()
    if any(q["kb_per_split"] > 1 and q["last_split_kb"] < q["kb_per_split"] for q in (p["dw1"], p["dw2"])):
        out.add("weight_multi_kblock_short_last")
    if p["dx"]["branch"] == "pick_splits":
        out.add("dx_pick_splits")
    if any(q["slices"] > 1 and q["kb_per_split"] > 1 for q in p.values()):
        out.add("slices_and_multi_kblock")
    if _cdiv(M, 128) > 16:
        out.add("finish_over_16_tiles")
    return out


def _bwd_workspace(M, Din, Dout, sms):
    """triad_project_tokens_bwd_workspace_bytes restated: [flag | gh | ln | tile partials | the largest product's
    fp32 split partials]; also the product whose partials set the size when one does strictly."""
    al = lambda v: _cdiv(v, 256) * 256                                                              # noqa: E731
    head = 256 + 2 * al(M * HIDDEN * 2) + al(_cdiv(M, 128) * 4 * HIDDEN * 4)
    part = {k: 256 + q["splits"] * q["rows"] * q["D"] * 4 for k, q in _bwd_plans(M, Din, Dout, sms).items()}
    top = max(part.values())
    winners = [k for k, v in part.items() if v == top]
    return head + top, winners[0] if len(winners) == 1 else None


# shapes at which dW1 (a 4-slice output, 6 k-blocks per item, the last split 5) and dW2 (2 k-blocks, the last split 1)
# set the workspace, so that their split counts are visible in it
PIN_SHAPES = [(3000, 2048, 16), (2600, 64, 512)]


def test_split_plan_restatement_matches_the_library():
    from triad_b200 import build, _lib
    build.build()
    lib = _lib.load()
    sms = _sms()
    revealed = {}
    for M, Din, Dout in [(c.M, c.Din, c.Dout) for c in BWD_CASES] + PIN_SHAPES:
        want, dominant = _bwd_workspace(M, Din, Dout, sms)
        assert lib.triad_project_tokens_bwd_workspace_bytes(M, Din, Dout) == want, (M, Din, Dout)
        if dominant:
            revealed.setdefault(dominant, []).append((M, Din, Dout))
    assert set(revealed) == {"dw2", "dw1", "dx"}, revealed


def test_every_regime_has_a_case():
    sms = _sms()
    seen = {}
    for c in BWD_CASES:
        for r in _regimes(c.M, c.Din, c.Dout, sms):
            seen.setdefault(r, []).append(c.name)
    missing = sorted(set(REGIMES) - set(seen))
    assert not missing, (missing, seen)


# ---- inputs ---------------------------------------------------------------------------------------------------------
EDGE_SCALES = {"small_var": (0.0, 2 ** -4, 2 ** -3, 2 ** -2, 2 ** -1, 1.0, 2.0, 4.0),
               "large_mean": (0.0, 32.0, 64.0, -32.0),
               "l2_zero": (0.0,)}
EDGE_B1 = {"small_var": 0.125, "large_mean": 96.0, "l2_zero": 0.125}


def _inputs(c, dev="cuda"):
    gen = torch.Generator(device=dev).manual_seed(20261022 + c.seed)

    def unif(n, lo, hi):
        return torch.rand(n, generator=gen, device=dev) * (hi - lo) + lo
    g, b, b2 = unif(HIDDEN, 0.5, 1.5), unif(HIDDEN, -0.3, 0.3), unif(c.Dout, -0.2, 0.2)
    w2 = (torch.randn(c.Dout, HIDDEN, generator=gen, device=dev) / math.sqrt(HIDDEN)).bfloat16()
    if c.exact:
        x = torch.randint(-3, 4, (c.M, c.Din), generator=gen, device=dev).bfloat16()
        w1 = (torch.randint(-1, 2, (HIDDEN, c.Din), generator=gen, device=dev) * 2.0 ** -6).bfloat16()
        b1 = torch.randint(-32, 33, (HIDDEN,), generator=gen, device=dev) * 2.0 ** -7
    else:
        x = torch.randn(c.M, c.Din, generator=gen, device=dev).bfloat16()
        w1 = (torch.randn(HIDDEN, c.Din, generator=gen, device=dev) / math.sqrt(c.Din)).bfloat16()
        b1 = unif(HIDDEN, -0.2, 0.2)
    rows = None
    if c.edge:
        # edge rows spread over the tiles: x = s e_j (s = 0: h = b1, a constant row), and for large_mean s (e_j - e_j')
        rows = torch.linspace(0, c.M - 1, min(c.M, 16), device=dev).round().long().unique()
        b1.fill_(EDGE_B1[c.edge])
        scales = EDGE_SCALES[c.edge]
        x[rows] = 0
        for i, r in enumerate(rows.tolist()):
            s = scales[i % len(scales)]
            x[r, (7 * r) % c.Din] = s
            if s < 0:
                x[r, (7 * r + 1) % c.Din] = -s
        if c.edge == "l2_zero":          # the constant rows' output is exactly 0
            b.zero_()
            b2.zero_()
    gy = (torch.randn(c.M, c.Dout, generator=gen, device=dev) * 0.1).bfloat16()
    return (x, w1, b1, g, b, w2, b2), gy, rows


# ---- checks ---------------------------------------------------------------------------------------------------------
def _ulp(v):
    """One bf16 ulp of the binade of |v| (fp64)."""
    return torch.ldexp(torch.ones_like(v), torch.frexp(v).exponent - 8)


def _bf16(v):
    """Round-to-nearest-even of fp64 values to bf16, exact (no detour through fp32)."""
    u = _ulp(v)
    return torch.round(v / u) * u


def _fwd_route(c):
    tiles = _cdiv(c.M, 128)
    return {"tiles": tiles, "last_tile_rows": c.M - 128 * (tiles - 1), "k_blocks": c.Din // 64,
            "halves": 2 if c.Dout > 256 else 1, "second_half_cols": c.Dout - 256 if c.Dout > 256 else None}


def _row_stats(h, eps):
    mu = h.mean(dim=1, keepdim=True)
    var = h.var(dim=1, unbiased=False, keepdim=True)
    rstd = (var + eps).rsqrt()
    return mu, var, rstd, (h - mu) * rstd


def _exact_row_sums(h, mu):
    """Rows whose fp32 sum of h and differences h - mean are exact: h on a common power-of-two grid (the smallest ulp
    among its non-zero elements) with the sum and 512 x the spread within 24 bits of it."""
    ulp = torch.where(h != 0, _ulp(h), torch.full_like(h, math.inf))
    grid = ulp.min(dim=1, keepdim=True).values.clamp(max=1.0)
    return ((h.abs().sum(dim=1, keepdim=True) / grid < 2.0 ** 24)
            & ((h - mu).abs().amax(dim=1, keepdim=True) * HIDDEN / grid < 2.0 ** 24))


def _check_forward(c, inp, t, got_off, got_on):
    x, w1, b1, g, b, w2, b2 = inp
    a, h, y, ln, out = (t[k].detach() for k in ("a", "h", "y", "ln", "out"))
    res = {}
    assert torch.isfinite(got_off).all() and torch.isfinite(got_on).all()
    mu, var, rstd, xh = _row_stats(h, c.eps)
    g64, b64 = g.double(), b.double()
    # h: bit-identical in exact cases; otherwise a may round either way within the first product's bound
    if c.exact:
        assert torch.equal(a.float().double(), a)                    # premise: a exact in fp32
        amb_h = torch.zeros_like(h, dtype=torch.bool)
    else:
        p1 = ((x.float() ** 2) @ (w1.float() ** 2).t()).sqrt().double() * 1.01
        e1 = ACC * math.sqrt(c.Din) * p1 + 2.0 ** -24 * a.abs()
        amb_h = _bf16(a - e1) != _bf16(a + e1)
        del p1, e1
    u_h = _ulp(h) * amb_h
    res["near_midpoint_h"] = int(amb_h.sum())
    # ln: the fp32 LayerNorm's deviation from y, then the near-midpoint ln
    exact_sum = _exact_row_sums(h, mu)
    shift = 2 * (u_h * (1 + xh.abs())).sum(dim=1, keepdim=True) * rstd / HIDDEN
    mean_term = torch.where(exact_sum, torch.zeros_like(rstd), LN_SUM * h.abs().mean(dim=1, keepdim=True) * rstd)
    xg = (xh * g64).abs()
    dy = LN_SUM * xg + mean_term * g64.abs() + LN_OP * (xg + b64.abs()) + g64.abs() * (1 + xh.abs()) * shift
    amb_ln = (_bf16(y - dy) != _bf16(y + dy)) | amb_h
    res["near_midpoint_ln"] = int(amb_ln.sum())
    dln = _ulp(ln) * amb_ln + u_h * rstd * g64.abs()
    del dy, xg, shift, u_h, amb_ln
    # the output's deviation before its rounding
    w2f = w2.float()
    p2 = ((ln.float() ** 2) @ (w2f ** 2).t()).sqrt().double()
    e_o = ACC * math.sqrt(HIDDEN) * p2 * 1.01 + 2.0 ** -23 * out.abs() + (dln.float() @ w2f.abs().t()).double() * 1.01
    del p2, dln
    go = got_off.double()
    if c.exact:
        lo, hi = _bf16(out - e_o), _bf16(out + e_o)
        bad = ((go < lo) | (go > hi)).nonzero()
        assert bad.numel() == 0, ("output", bad[:8].tolist(), go[tuple(bad[0])].item(), out[tuple(bad[0])].item())
        near = int((lo != hi).sum())
        assert near <= max(0.25 * out.numel(), 8), near            # the check is not vacuous
        res["near_midpoint_out"] = near
        res["flipped_out"] = int((go != _bf16(out)).sum())
        del lo, hi
    else:
        err = (go - out).norm(dim=1)
        bound = 2.0 ** -9 * out.norm(dim=1) + (1 + 2.0 ** -9) * e_o.norm(dim=1)
        ratio = err / bound
        worst = int(ratio.argmax())
        assert (err <= bound).all(), ("row", worst, err[worst].item(), bound[worst].item())
        res["out_row_over_bound"] = ratio.max().item()
    del e_o
    # normalize=True against the fp64 normalisation of the kernel's own o
    n = go / go.norm(dim=1, keepdim=True).clamp(min=1e-12)
    tau = (c.Dout + 8) * 2.0 ** -24
    lo, hi = _bf16(n - tau * n.abs()), _bf16(n + tau * n.abs())
    gn = got_on.double()
    bad = ((gn < lo) | (gn > hi)).nonzero()
    assert bad.numel() == 0, ("normalized", bad[:8].tolist())
    res["near_midpoint_normalized"] = int((lo != hi).sum())
    return res, (mu, var)


def _edge_report(c, rows, mu, var, got_off, got_on):
    """What the edge rows are, asserted so that each case exercises its edge."""
    v, m = var[rows, 0], mu[rows, 0]
    if c.edge == "small_var":
        r = (v / c.eps).tolist()
        assert min(r) == 0.0                                        # a constant row: rstd = 1/sqrt(eps)
        assert any(0 < q < 0.1 for q in r) and any(0.1 <= q <= 1.0 for q in r), r   # below eps, and near it
        return {"var_over_eps": sorted(round(q, 4) for q in r)}
    if c.edge == "large_mean":
        live = v > 0
        ratio = (m[live] ** 2 / v[live])
        assert (v == 0).any() and live.sum() >= 3 and ratio.min().item() >= 1e4, ratio.tolist()
        return {"mean2_over_var_min": ratio.min().item(), "var_zero_rows": int((v == 0).sum())}
    # l2_zero: the constant rows' output is exactly zero, every other row's is not
    zero = torch.zeros(c.M, dtype=torch.bool, device=got_off.device)
    zero[rows] = True
    assert (got_off[zero] == 0).all() and (got_on[zero] == 0).all()
    assert (got_off[~zero].float().norm(dim=1) > 0).all()
    return {"zero_rows": int(zero.sum())}


def _block_norms(t, br, bc):
    t = t.reshape(-1, t.shape[-1]) if t.dim() > 1 else t.reshape(1, -1)
    R, C = t.shape
    t = torch.nn.functional.pad(t, (0, (-C) % bc, 0, (-R) % br))
    return t.reshape(t.shape[0] // br, br, t.shape[1] // bc, bc).square().sum(dim=(1, 3)).sqrt()


def _check_backward(got, ref, cf):
    res = {}
    for name, k, r, f in zip(NAMES, got, ref, cf):
        assert torch.isfinite(k).all(), name
        k, r = k.detach().double().reshape(r.shape), r.detach()
        rnorm = r.norm().clamp(min=1e-30)
        ek = ((k - r).norm() / rnorm).item()
        ec = ((f.detach().double().reshape(r.shape) - r).norm() / rnorm).item()
        assert ek <= SLACK * ec + ABS_SLACK, (name, ek, ec)
        br, bc = BLOCKS[name]
        err, want = _block_norms(k - r, br, bc), _block_norms(r, br, bc)
        bound = GRAD_TOL[name] * want.clamp(min=1e-3 * rnorm.item())
        ratio = err / bound
        worst = divmod(int(ratio.argmax()), ratio.shape[1])
        assert (err <= bound).all(), (name, "block", worst, ratio.max().item())
        res[name] = {"block_over_bound": ratio.max().item(), "frob": ek, "closed_form_frob": ec}
    return res


def _report(c, kind, payload):
    print(json.dumps({"case": c.name, "check": kind, "M": c.M, "Din": c.Din, "Dout": c.Dout, **payload}))


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_head_against_fp64(case):
    from triad_b200.producers import project_tokens, project_tokens_bwd
    from tests.test_gpu_projection_backward import _closed_form
    c = case
    torch.cuda.reset_peak_memory_stats()
    inp, gy, rows = _inputs(c)
    x, w1, b1, g, b, w2, b2 = inp
    leaves, t = head_fp64(*inp, c.eps, requires_grad=c.bwd)
    if c.fwd:
        got_off = project_tokens(x, w1, b1, g, b, c.eps, w2, b2, normalize=False)
        got_on = project_tokens(x, w1, b1, g, b, c.eps, w2, b2, normalize=True)
        res, (mu, var) = _check_forward(c, inp, t, got_off, got_on)
        if c.edge:
            res["edge"] = _edge_report(c, rows, mu, var, got_off, got_on)
        del mu, var, got_off, got_on
        _report(c, "forward", {"route": _fwd_route(c), **res, "peak_mem_gb": torch.cuda.max_memory_allocated() / 1e9})
    if c.bwd:
        if c.edge:                      # the backward's rstd takes eps too: the edge rows must be what they claim
            _, var, _, _ = _row_stats(t["h"].detach(), c.eps)
            assert var[rows].min().item() == 0.0
            del var
        t["out"].backward(gy.double())
        ref = tuple(v.grad for v in leaves)
        del t, leaves
        got = project_tokens_bwd(x, w1, b1, g, b, c.eps, w2, gy, (True,) * 7)
        cf = _closed_form(x, w1, b1, g, b, w2, c.eps, gy)
        res = _check_backward(got, ref, cf)
        worst = max(v["block_over_bound"] for v in res.values())
        _report(c, "backward", {"route": {**_bwd_plans(c.M, c.Din, c.Dout, _sms()), "finish_tiles": _cdiv(c.M, 128),
                                          "regimes": sorted(_regimes(c.M, c.Din, c.Dout, _sms()))},
                                "worst_over_bound": worst, "grads": res,
                                "peak_mem_gb": torch.cuda.max_memory_allocated() / 1e9})
