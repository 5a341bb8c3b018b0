"""Backward of the projection head (triad_project_tokens_bwd) and of patch dropout (triad_patch_expand).

The head's seven gradients are checked against an fp64 autograd reference of the autocast recipe (bf16 weights and
input, h and the LayerNorm output rounded to bf16 as the forward rounds them; the rounding passes gradients straight
through), next to the torch closed form the kernels replaced: per gradient, the kernels may not be further from fp64
than that closed form.  CPU tier: argument validation of the new entry points."""
import ctypes

import pytest
import torch

from triad_b200.producers import ProjectionHead, patch_dropout, patch_expand, project_tokens_bwd
from tests.helpers import head_fp64_grads, rel_err

NAMES = ("dx", "dw1", "db1", "dg", "db", "dw2", "db2")
ALL = (True,) * 7
# Absolute bars against fp64, relative Frobenius error:
#   dx        bf16 output of gh . W1 with gh rounded to bf16: a few bf16 ulps (2^-9 = 2e-3 each)
#   dw1, dw2  fp32 sums over tokens of products of bf16-rounded operands (gh, ln): the operand rounding dominates
#   vectors   fp32 sums of fp32 terms (db2 sums the bf16 gy exactly as given)
ABS_BAR = {"dx": 1e-2, "dw1": 5e-3, "db1": 1e-3, "dg": 1e-3, "db": 1e-3, "dw2": 5e-3, "db2": 1e-4}
# Against the closed form: err(kernels) <= SLACK * err(closed form) + ABS_SLACK.  The kernels' weight gradients stay
# fp32 and gln is not rounded to bf16, so they are usually well below; dx and db2 round like the closed form and
# differ from it only in summation order.
SLACK, ABS_SLACK = 1.25, 2e-5


def _head(Din, Dout, seed):
    torch.manual_seed(seed)
    head = ProjectionHead(Din, Dout).cuda()
    with torch.no_grad():
        head.layer_norm.weight.uniform_(0.5, 1.5)
        head.layer_norm.bias.uniform_(-0.3, 0.3)
        head.projection1.bias.uniform_(-0.2, 0.2)
        head.projection2.bias.uniform_(-0.2, 0.2)
    return head


def _params(head):
    return (head.projection1.weight, head.projection1.bias, head.layer_norm.weight, head.layer_norm.bias,
            head.projection2.weight, head.projection2.bias)


def _closed_form(x, w1, b1, g, b, w2, eps, gy):
    """The torch closed form this backward replaced (bf16 library GEMMs, fp32 LayerNorm algebra)."""
    Din = x.shape[-1]
    x2 = x.reshape(-1, Din)
    gy2 = gy.reshape(-1, gy.shape[-1]).to(torch.bfloat16)
    w1b, w2b = w1.to(torch.bfloat16), w2.to(torch.bfloat16)
    h = (x2 @ w1b.t() + b1.to(torch.bfloat16)).float()
    mu = h.mean(dim=1, keepdim=True)
    rstd = torch.rsqrt(h.var(dim=1, unbiased=False, keepdim=True) + eps)
    xh = (h - mu) * rstd
    ln = (xh * g.float() + b.float()).to(torch.bfloat16)
    gw2 = gy2.t() @ ln
    gb2 = gy2.float().sum(dim=0)
    gln = (gy2 @ w2b).float()
    gg = (gln * xh).sum(dim=0)
    gb = gln.sum(dim=0)
    gxh = gln * g.float()
    gh = (gxh - gxh.mean(dim=1, keepdim=True) - xh * (gxh * xh).mean(dim=1, keepdim=True)) * rstd
    ghb = gh.to(torch.bfloat16)
    gw1 = ghb.t() @ x2
    gb1 = gh.sum(dim=0)
    gx = (ghb @ w1b).view_as(x)
    return gx, gw1.float(), gb1, gg, gb, gw2.float(), gb2


SHAPES = [(4, 250, 768, 512), (3, 77, 768, 512), (2, 256, 384, 512), (1, 5, 64, 64), (2, 130, 1024, 256), (1, 1, 128, 16),
          (2, 300, 768, 320),
          (1, 1, 768, 512), (1, 127, 384, 64), (1, 129, 1536, 16), (3, 43, 1024, 320), (1, 129, 64, 512), (1, 127, 1536, 512)]


@pytest.mark.gpu
@pytest.mark.parametrize("B,N,Din,Dout", SHAPES)
def test_head_backward_against_fp64(B, N, Din, Dout):
    head = _head(Din, Dout, Din + N + Dout)
    x = torch.randn(B, N, Din, device="cuda").bfloat16()
    gy = (torch.randn(B, N, Dout, device="cuda") * 0.1).bfloat16()
    w1, b1, g, b, w2, b2 = (t.detach() for t in _params(head))
    eps = head.layer_norm.eps
    got = project_tokens_bwd(x, w1, b1, g, b, eps, w2, gy, ALL)
    cf = _closed_form(x, w1, b1, g, b, w2, eps, gy)
    ref = head_fp64_grads(x, w1, b1, g, b, w2, b2, eps, gy)
    assert got[0].shape == x.shape and got[0].dtype == torch.bfloat16
    assert got[1].shape == (512, Din) and got[5].shape == (Dout, 512) and got[6].shape == (Dout,)
    for name, k, c, r in zip(NAMES, got, cf, ref):
        ek, ec = rel_err(k, r), rel_err(c, r)
        assert torch.isfinite(k).all(), name
        assert ek <= SLACK * ec + ABS_SLACK, (name, ek, ec)
        assert ek < ABS_BAR[name], (name, ek)


@pytest.mark.gpu
def test_head_backward_is_deterministic():
    head = _head(768, 512, 1)
    x = torch.randn(8, 250, 768, device="cuda").bfloat16()
    gy = torch.randn(8, 250, 512, device="cuda").bfloat16()
    args = [t.detach() for t in _params(head)]
    w1, b1, g, b, w2, _ = args
    a = project_tokens_bwd(x, w1, b1, g, b, 1e-5, w2, gy, ALL)
    c = project_tokens_bwd(x, w1, b1, g, b, 1e-5, w2, gy, ALL)
    for name, u, v in zip(NAMES, a, c):
        assert torch.equal(u, v), name


@pytest.mark.gpu
def test_needs_input_grad_subsets_match_the_full_call():
    head = _head(384, 256, 2)
    x = torch.randn(3, 90, 384, device="cuda").bfloat16()
    gy = torch.randn(3, 90, 256, device="cuda").bfloat16()

    def run(x_grad, w_grad):
        head.zero_grad(set_to_none=True)
        for t in _params(head):
            t.requires_grad_(w_grad)
        xi = x.clone().requires_grad_(x_grad)
        head(xi).backward(gy)
        return xi.grad, [t.grad for t in _params(head)]

    gx_full, gw_full = run(True, True)
    gx_frozen, gw = run(False, True)                 # frozen encoder: no dx
    assert gx_frozen is None
    for u, v in zip(gw, gw_full):
        assert torch.equal(u, v)
    gx, gw_none = run(True, False)                   # frozen head: no weight gradients
    assert all(t is None for t in gw_none)
    assert torch.equal(gx, gx_full)
    for t in _params(head):
        t.requires_grad_(True)
    # the raw call with single outputs
    w1, b1, g, b, w2, _ = (t.detach() for t in _params(head))
    full = project_tokens_bwd(x, w1, b1, g, b, head.layer_norm.eps, w2, gy, ALL)
    for i in range(7):
        need = tuple(j == i for j in range(7))
        one = project_tokens_bwd(x, w1, b1, g, b, head.layer_norm.eps, w2, gy, need)
        assert all(t is None for j, t in enumerate(one) if j != i)
        assert torch.equal(one[i], full[i]), NAMES[i]


@pytest.mark.gpu
def test_backward_has_no_host_synchronisation():
    head = _head(768, 512, 3)
    xa = torch.randn(4, 64, 768, device="cuda").bfloat16().requires_grad_()
    xv = torch.randn(4, 96, 768, device="cuda").bfloat16().requires_grad_()
    torch.manual_seed(4)
    y = patch_dropout(head(xv), 0.5)             # the forward sizes its output on the host; the backward must not sync
    loss = y.float().square().sum() + head(xa).float().sum()
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        loss.backward()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    assert torch.isfinite(xv.grad.float()).all() and torch.isfinite(xa.grad.float()).all()


def _expand_formula(gy, keep, n):
    """The indexing formula of the compaction's backward (what patch_dropout's backward computed before)."""
    B, L, D = gy.shape
    pos = keep.long().cumsum(dim=1) - 1
    gx = gy.new_zeros(B, n, D)
    bi, ni = keep.nonzero(as_tuple=True)
    gx[bi, ni] = gy[bi, pos[bi, ni]]
    return gx


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,B,N,D", [(torch.bfloat16, 7, 256, 512), (torch.float32, 5, 33, 12), (torch.bfloat16, 3, 1030, 64)])
def test_patch_expand_matches_the_indexing_formula(dtype, B, N, D):
    torch.manual_seed(N)
    for rate in (0.1, 0.5, 0.9):
        keep = torch.rand(B, N, device="cuda") >= rate
        keep[0] = False                                          # an image with every patch dropped
        longest = int(keep.sum(dim=1).max().item())
        for max_len in (longest, longest + 5):                   # and rows behind the longest kept list
            gy = torch.randn(B, max_len, D, device="cuda").to(dtype)
            assert torch.equal(patch_expand(gy, keep, N), _expand_formula(gy, keep, N)), (rate, max_len)


@pytest.mark.gpu
def test_patch_dropout_backward_matches_the_indexing_formula():
    x = torch.randn(6, 256, 64, device="cuda").bfloat16().requires_grad_()
    torch.manual_seed(9)
    y = patch_dropout(x, 0.3)
    gy = torch.randn_like(y)
    y.backward(gy)
    torch.manual_seed(9)
    keep = torch.bernoulli(torch.ones(6, 256, device="cuda", dtype=x.dtype) * 0.7).bool()
    assert torch.equal(x.grad, _expand_formula(gy, keep, 256))


def _loop_patch_dropout(x, drop_rate):
    """The reference's patch dropout (model.py:283-307), restated."""
    B, N, D = x.shape
    keep = torch.bernoulli(torch.ones(B, N, device=x.device, dtype=x.dtype) * (1 - drop_rate)).bool()
    kept = [x[i][keep[i]] for i in range(B)]
    m = max(t.size(0) for t in kept)
    return torch.stack([torch.cat([t, torch.zeros(m - t.size(0), D, dtype=x.dtype, device=x.device)]) for t in kept])


@pytest.mark.gpu
def test_chain_head_dropout_av_loss_matches_torch_nn():
    from triad_b200 import TriadHotPath
    torch.manual_seed(21)
    B, Na, Nv, Din = 8, 40, 64, 768
    ha, hv = _head(Din, 512, 5), _head(Din, 512, 6)
    ra, rv = _head(Din, 512, 7), _head(Din, 512, 8)
    ra.load_state_dict(ha.state_dict())
    rv.load_state_dict(hv.state_dict())
    xa = torch.randn(B, Na, Din, device="cuda").bfloat16()
    xv = torch.randn(B, Nv, Din, device="cuda").bfloat16()
    loss_mod = TriadHotPath().cuda()
    loss_mod.triad_regularizers = False

    xa1, xv1 = xa.clone().requires_grad_(), xv.clone().requires_grad_()
    torch.manual_seed(33)
    va = patch_dropout(hv(xv1), 0.25)
    loss_mod.forward_features_av(ha(xa1), va)[0].backward()

    def nn_head(h, x):
        with torch.autocast("cuda", dtype=torch.bfloat16):
            return h.projection2(h.layer_norm(h.projection1(x)))
    xa2, xv2 = xa.clone().requires_grad_(), xv.clone().requires_grad_()
    torch.manual_seed(33)
    vb = _loop_patch_dropout(nn_head(rv, xv2), 0.25)
    loss_mod.forward_features_av(nn_head(ra, xa2), vb)[0].backward()

    assert va.shape == vb.shape
    assert rel_err(xa1.grad, xa2.grad) < 3e-2 and rel_err(xv1.grad, xv2.grad) < 3e-2
    for mine, ref in ((ha, ra), (hv, rv)):
        for (n, a), (_, b) in zip(mine.named_parameters(), ref.named_parameters()):
            assert rel_err(a.grad, b.grad) < 3e-2, n


def test_backward_entry_points_validate_arguments_without_gpu():
    """triad_project_tokens_bwd and triad_patch_expand reject bad arguments before any CUDA call."""
    from triad_b200 import build, _lib
    build.build()
    lib = _lib.load()
    E = {"arg": -1, "shape": -2, "align": -3, "ws": -4, "unsupported": -7}
    null = None
    one = ctypes.c_void_p(16)
    odd = ctypes.c_void_p(24)
    f = lib.triad_project_tokens_bwd

    def call(x=one, w1=one, gy=one, M=256, Din=768, Dout=512, dx=one, dw1=one, db1=one, ws=one, ws_bytes=1 << 40):
        return f(x, w1, one, one, one, 1e-5, one, gy, M, Din, Dout, dx, dw1, db1, one, one, one, one, ws, ws_bytes, null)

    assert call(x=null) == E["arg"]
    assert call(gy=null) == E["arg"]
    assert call(ws=null) == E["arg"]
    assert call(M=0) == E["shape"]
    assert call(Din=96) == E["unsupported"]                      # Din % 64
    assert call(Dout=520) == E["unsupported"]                    # Dout > 512
    assert call(Dout=40) == E["unsupported"]                     # Dout % 16
    assert call(gy=odd) == E["align"]
    assert call(dw1=odd) == E["align"]
    assert call(db1=ctypes.c_void_p(18)) == E["align"]
    need = lib.triad_project_tokens_bwd_workspace_bytes(256, 768, 512)
    assert need >= 256 * 512 * 2 * 2                             # the bf16 hidden gradient and LayerNorm output
    assert call(ws_bytes=need - 1) == E["ws"]
    assert lib.triad_project_tokens_bwd_workspace_bytes(0, 768, 512) == 0
    e = lib.triad_patch_expand
    assert e(null, one, 2, 8, 64, 2, 4, one, null) == E["arg"]
    assert e(one, null, 2, 8, 64, 2, 4, one, null) == E["arg"]
    assert e(one, one, 2, 8, 4, 2, 4, one, null) == E["shape"]    # row bytes % 16
    assert e(one, one, 0, 8, 64, 2, 4, one, null) == E["shape"]
    assert e(odd, one, 2, 8, 64, 2, 4, one, null) == E["align"]
    assert e(one, one, 2, 60000, 64, 2, 4, one, null) == E["unsupported"]
