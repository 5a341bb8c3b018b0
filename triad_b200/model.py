"""Drop-in replacements for the similarity / aggregation / loss methods of the reference's
``MultiModalModel`` (src/model.py:355-392, :430-472, :490-514, :544-593).

``TriadSimilarityMixin`` keeps the reference's method names, positional arguments and return
arities, so ``forward_audio_visual`` (model.py:487-488), ``forward_text_visual`` (:607-608) and
the trainer (train.py:745,758,954,969) run unchanged on top of it:

    class MultiModalModel(TriadSimilarityMixin, nn.Module): ...   # see INTEGRATION.md

``self`` only has to provide what the reference's methods read: ``self.temperature`` (0-dim fp32
nn.Parameter, model.py:348) and ``patch_sparsity_threshold`` / ``patch_sparsity_weight``.

One deliberate difference: the reference returns the dense ``token_sims`` tensor
(B,B,Nq,Nv) — 16.8 GB at the B=256 training shape.  The fused path never builds it; the second
return value is a ``TokenSims`` handle that carries the saved argmax indices and the fp32 clip
matrix, has the reference tensor's ``.shape`` / ``.dtype`` / ``.device``, and can
``.materialize()`` the dense tensor on demand (visualisation, tests, small batches).  The loss
methods accept that handle and evaluate the reference's regularisers from the embeddings it
carries (regularizers.py); given a dense tensor instead, only the contrastive part — which
never needed token_sims — is computed from ``clip_sims``.
"""
from __future__ import annotations

from collections.abc import Mapping
from typing import Dict, Optional, Tuple

import torch

from . import ops
from . import _lib as _lib_flags


class TokenSims:
    """Stand-in for the reference's (Bq,Bv,Nq,Nv) token-similarity tensor."""

    def __init__(self, q, v, temperature, scale, mask, clip_f32, idx, prefix):
        self.q, self.v, self.temperature = q, v, temperature
        self.row_scale, self.mask = scale, mask
        self.clip = clip_f32            # fp32 (Bq,Bv), attached to the autograd graph
        self.idx_t = idx                # [Bv, Bq*nq_pad] uint8/uint16 (library layout)
        self.prefix = prefix
        self.clip_out = clip_f32        # what compute_all_similarities_* returned as clip_sims (set by the caller)
        self.packed = False
        self.fwd_flags = 0
        self.nonneg = None              # (N, sums, lo) when the forward also produced the dense regulariser's gradient
        self.shape = torch.Size((q.shape[0], v.shape[0], q.shape[1], v.shape[1]))
        self.dtype = q.dtype
        self.device = q.device

    def take_nonneg(self, lo: float):
        """(N, sums) of the dense regulariser if the forward produced them for this clamp floor — handed over ONCE
        (N is gigabytes: the handle drops its reference), else None."""
        if self.nonneg is None or self.nonneg[2] != lo:
            return None
        N, sums, _ = self.nonneg
        self.nonneg = None
        return N, sums

    def argmax(self) -> torch.Tensor:
        """(Bq,Bv,Nq) int64 in the reference's layout: torch.max(token_sims, dim=3)[1].

        When padded tokens were dropped from the training forward (``packed``), their winners — which
        the reference computes although nothing depends on them — are produced here by one forward over
        all rows (inspection / parity tests only; not on the training path)."""
        idx = self.idx_t
        if self.packed:
            T = ops.temperature_tensor(self.temperature, self.device)
            _, idx = ops.maxmean_fwd(self.q.detach(), self.v.detach(), self.row_scale, T, want_idx=True,
                                     flags=self.fwd_flags & ~_lib_flags.FWD_PACK_ROWS)
        return ops.idx_to_reference_layout(idx, self.shape[0], self.shape[2])

    def materialize(self) -> torch.Tensor:
        """Dense token_sims exactly as the reference builds it (model.py:384-387).  Debug /
        visualisation aid for small batches; not used by the training path."""
        Bq, Bv = self.shape[0], self.shape[1]
        af = self.q.unsqueeze(1).expand(-1, Bv, -1, -1)
        vf = self.v.unsqueeze(0).expand(Bq, -1, -1, -1)
        return torch.matmul(af, vf.transpose(2, 3)) * self.temperature

    def __repr__(self):
        return f"TokenSims(shape={tuple(self.shape)}, dtype={self.dtype}, device={self.device}, fused)"


class LazyStats(Mapping):
    """The statistics dictionary of model.py:463-470, filled on first access.

    The reference pays five ``.item()`` device->host syncs per loss call to build this dict even
    when nobody looks at it.  Here the six values live in one small device tensor until a key is
    actually read (wandb logging, prints); the training step itself stays asynchronous, so the
    backward kernels can be queued while the forward is still running.

    A read-only ``Mapping`` (not a ``dict`` subclass: C fast paths such as ``json.dumps`` or ``pickle`` read a
    dict's storage directly and would see it empty).  ``wandb_dict.update(stats)``, ``stats[key]``,
    ``key in stats``, ``stats.keys()``, ``dict(stats)`` and ``**stats`` work as with the reference's dict;
    ``to_dict()`` / pickling / deepcopy give a plain dict."""

    __slots__ = ("_pending", "_values")

    def __init__(self, sums: torch.Tensor, B: int, prefix: str):
        self._pending = (sums, B, prefix)
        self._values = None

    def _fill(self) -> Dict[str, float]:
        if self._values is None:
            sums, B, prefix = self._pending
            self._values = _stats_from_sums(sums, B, prefix)
            self._pending = None
        return self._values

    def __getitem__(self, k):
        return self._fill()[k]

    def __iter__(self):
        return iter(self._fill())

    def __len__(self):
        return len(self._fill())

    def __repr__(self):
        return repr(self._fill())

    def to_dict(self) -> Dict[str, float]:
        return dict(self._fill())

    def copy(self) -> Dict[str, float]:
        return self.to_dict()

    def __reduce__(self):
        return (dict, (self.to_dict(),))

    def __deepcopy__(self, memo):
        return self.to_dict()


def _stats_from_sums(sums: torch.Tensor, B: int, prefix: str) -> Dict[str, float]:
    """model.py:435-450 / :553-568 from the kernel's fp64 sums; ONE device->host copy instead of
    the reference's five .item() calls.  B = 1 has no off-diagonal entry: the negative statistics, the separation and
    the hardest negative are NaN (where the reference's max over an empty tensor raises)."""
    s = sums.tolist()
    n_off = B * B - B
    pos_mean = s[1] / B
    neg_mean = s[3] / n_off if n_off else float("nan")
    pos_var = (s[2] - B * pos_mean * pos_mean) / (B - 1) if B > 1 else float("nan")
    neg_var = (s[4] - n_off * neg_mean * neg_mean) / (n_off - 1) if n_off > 1 else float("nan")
    return {
        f"{prefix}_pos_sim_mean": pos_mean,
        f"{prefix}_pos_sim_std": max(pos_var, 0.0) ** 0.5 if pos_var == pos_var else pos_var,
        f"{prefix}_neg_sim_mean": neg_mean,
        f"{prefix}_neg_sim_std": max(neg_var, 0.0) ** 0.5 if neg_var == neg_var else neg_var,
        f"{prefix}_separation": pos_mean - neg_mean,
        f"{prefix}_hardest_negative": s[5] if n_off else float("nan"),
    }


_zeros: Dict[torch.device, torch.Tensor] = {}


def _zero_scalar(device) -> torch.Tensor:
    """A constant fp32 zero on `device` (the 0.01*l_smooth slot when the regularisers are off): made once, not per step."""
    z = _zeros.get(device)
    if z is None:
        z = _zeros[device] = torch.zeros((), dtype=torch.float32, device=device)
    return z


class TriadSimilarityMixin:
    """Provides compute_all_similarities_{av,tv}, compute_contrastive_loss_{av,tv} and
    compute_similarity_matrix with the reference's signatures."""

    #: forwarded to triad_maxmean_fwd (tests use it to pin a kernel variant)
    triad_fwd_flags: int = 0
    #: drop zero-weight (padded) text tokens before the GEMM (bf16 tensor-core path); their argmax entries are
    #: then only produced on demand by TokenSims.argmax()
    triad_pack_masked_rows: bool = True
    #: evaluate the reference's regularisation terms (model.py:394-428, :516-542) in the loss methods
    triad_regularizers: bool = True

    # -- similarities -----------------------------------------------------------------------
    def _similarities(self, q_feats, visual_feats, attention_mask, prefix):
        if q_feats.dim() != 3 or visual_feats.dim() != 3:
            raise ValueError("expected (B,N,D) embeddings")
        ops._require_cuda(q_feats, visual_feats, attention_mask)
        if q_feats.dtype != visual_feats.dtype or q_feats.dtype not in (torch.float32, torch.bfloat16):
            raise TypeError(f"triad_b200 supports float32 and bfloat16 embeddings of one dtype, got "
                            f"{q_feats.dtype} / {visual_feats.dtype}")
        Bq, Nq, _ = q_feats.shape
        scale = ops.row_scale(attention_mask, Bq, Nq, q_feats.device)
        flags = int(self.triad_fwd_flags)
        # padded text tokens (weight 0, model.py:509-512) are dropped before the tensor cores
        if attention_mask is not None and q_feats.dtype == torch.bfloat16 and self.triad_pack_masked_rows:
            flags |= _lib_flags.FWD_PACK_ROWS
        # With the reference's regularisers on, the loss call that follows needs N = dL/d<q,v> of the dense
        # non-negative-pressure term over the very same similarity tiles (model.py:411-412 / :525-526): one pass
        # produces both (regularizers.merged_forward_ok); all rows take part there, so no packing.
        from . import regularizers as R
        nonneg_lo = None
        if (bool(getattr(self, "triad_regularizers", True)) and torch.is_grad_enabled()
                and (q_feats.requires_grad or visual_feats.requires_grad or self.temperature.requires_grad)
                and R.merged_forward_ok(q_feats, visual_feats)):
            nonneg_lo = -60.0 if attention_mask is None else -20.0
            bwd_pack = bool(flags & _lib_flags.FWD_PACK_ROWS)
            flags &= ~_lib_flags.FWD_PACK_ROWS
        clip, idx, N, nsums = ops.MaxMeanSimilarity.apply(q_feats, visual_feats, self.temperature, scale, flags,
                                                          attention_mask is None, nonneg_lo,
                                                          nonneg_lo is not None and bwd_pack)
        handle = TokenSims(q_feats, visual_feats, self.temperature, scale, attention_mask, clip, idx, prefix)
        handle.packed = bool(flags & _lib_flags.FWD_PACK_ROWS)
        handle.fwd_flags = flags
        if N is not None:
            handle.nonneg = (N, nsums, nonneg_lo)
        # The reference's clip_sims dtype: bf16 for AV under autocast (mean of bf16 maxima,
        # model.py:391), fp32 for TV (mask.float() promotes, model.py:509-512) and for fp32 inputs.
        out = clip.to(q_feats.dtype) if attention_mask is None else clip
        handle.clip_out = out
        return out, handle

    def compute_all_similarities_av(self, audio_feats, visual_feats):
        """(clip_sims (B,B), token_sims handle) — model.py:370-392."""
        return self._similarities(audio_feats, visual_feats, None, "av")

    def compute_all_similarities_tv(self, text_feats, visual_feats, attention_mask):
        """(clip_sims (B,B), token_sims handle) — model.py:490-514."""
        return self._similarities(text_feats, visual_feats, attention_mask, "tv")

    # -- losses -----------------------------------------------------------------------------
    def _loss_head(self, clip_sims, token_sims, prefix, with_calibration):
        """(contrastive, l_cal or None, contrastive + l_cal or None, stats).

        The loss is computed from the ``clip_sims`` argument, as in the reference.  When that argument is the very
        tensor compute_all_similarities_* returned next to the handle, the handle's fp32 copy of the same matrix
        is used instead of its bf16 rounding (the reference's log_softmax runs in fp32 under autocast; the
        unrounded input is the more accurate of the two and keeps one autograd path).  Anything else — a scaled,
        detached or otherwise edited matrix — is honoured as given."""
        clip = clip_sims
        if isinstance(token_sims, TokenSims) and (clip_sims is token_sims.clip_out or clip_sims is token_sims.clip):
            clip = token_sims.clip
        if not isinstance(clip, torch.Tensor) or clip.dim() != 2:
            raise ValueError("clip_sims must be the (B,B) clip-similarity matrix")
        ops._require_cuda(clip)
        B = clip.shape[0]
        T = self.temperature if with_calibration else None
        if B <= ops.HEAD_MAX_B:
            con, cal, tot, sums = ops.ContrastiveHead.apply(clip, T)
            if not with_calibration:
                cal = tot = None
        else:                                   # very large single-device batches: the block-wise kernels
            con, sums = ops.SymmetricInfoNCE.apply(clip)
            cal = self._temperature_calibration() if with_calibration else None
            tot = con + cal if with_calibration else None
        return con, cal, tot, LazyStats(sums, B, prefix)

    def _temperature_calibration(self) -> torch.Tensor:
        """20 * relu(-log T)^2 — the l_cal term of model.py:420-427 (a scalar on the parameter)."""
        return 20.0 * torch.clamp(-torch.log(self.temperature), min=0) ** 2

    def _dense_terms_enabled(self, token_sims) -> bool:
        return bool(getattr(self, "triad_regularizers", True)) and isinstance(token_sims, TokenSims)

    def compute_regularization_losses_av(self, token_sims):
        """(reg, 0.01*l_smooth) — model.py:410-428: 20*l_cal + 0.15*mean(clamp(S,-60,0)^2) + 0.01*l_smooth."""
        return self._regularization_av(token_sims, None)

    def _regularization_av(self, token_sims, l_cal):
        """compute_regularization_losses_av with the calibration term already evaluated by the fused head."""
        from . import regularizers as R
        tok = token_sims
        l_nonneg = R.nonneg_pressure(tok.q, tok.v, self.temperature, -60.0, precomputed=tok.take_nonneg(-60.0))
        l_smooth = R.temporal_smoothness(tok.q, tok.v, self.temperature)
        if l_cal is None:
            l_cal = self._temperature_calibration()
        reg = l_cal + 0.15 * l_nonneg + 0.01 * l_smooth
        return reg, 0.01 * l_smooth

    def compute_regularization_losses_tv(self, token_sims):
        """reg — model.py:516-542: 0.15*mean(clamp(S,-20,0)^2) + patch_sparsity_weight*sparsity."""
        from . import regularizers as R
        tok = token_sims
        l_nonneg = R.nonneg_pressure(tok.q, tok.v, self.temperature, -20.0, precomputed=tok.take_nonneg(-20.0))
        sparsity = R.patch_sparsity(tok.q, tok.v, self.temperature, self.patch_sparsity_threshold)
        return 0.15 * l_nonneg + self.patch_sparsity_weight * sparsity

    def compute_contrastive_loss_av(self, clip_sims, token_sims):
        """(total, contrastive, reg, 0.01*l_smooth, stats) — model.py:430-472.

        ``token_sims`` is the TokenSims handle of compute_all_similarities_av; the regularisers are
        evaluated from the embeddings it carries (regularizers.py).  With ``self.triad_regularizers =
        False`` (or a dense tensor in place of the handle) only the contrastive loss and the scalar
        temperature-calibration term are computed — the fused max-mean + InfoNCE path on its own, which
        is what BASELINE.json's metric times."""
        contrastive, l_cal, con_plus_cal, stats = self._loss_head(clip_sims, token_sims, "av", True)
        if self._dense_terms_enabled(token_sims):
            reg, smooth = self._regularization_av(token_sims, l_cal)
            return contrastive + reg, contrastive, reg, smooth, stats
        return con_plus_cal, contrastive, l_cal, _zero_scalar(contrastive.device), stats

    def compute_contrastive_loss_tv(self, clip_sims, token_sims):
        """(total, stats) — model.py:544-593 (see compute_contrastive_loss_av for the regulariser switch)."""
        contrastive, _, _, stats = self._loss_head(clip_sims, token_sims, "tv", False)
        if self._dense_terms_enabled(token_sims):
            return contrastive + self.compute_regularization_losses_tv(token_sims), stats
        return contrastive, stats

    # -- per-pair normalised similarity (viz / forward()) -------------------------------------
    def compute_similarity_matrix(self, feats1, feats2):
        """(B,N1,N2) = T * <normalize(f1), normalize(f2)> — model.py:355-368 (inference helper,
        no autograd)."""
        from . import _lib
        lib = _lib.load()
        f1 = feats1.detach().float().contiguous()
        f2 = feats2.detach().float().contiguous()
        B, N1, D = f1.shape
        N2 = f2.shape[1]
        T = ops.temperature_tensor(self.temperature, f1.device)
        out = torch.empty(B, N1, N2, dtype=torch.float32, device=f1.device)
        with ops._on(f1):
            _lib.check(lib.triad_similarity_matrix(f1.data_ptr(), f2.data_ptr(), T.data_ptr(), B, N1, N2, D,
                                                   out.data_ptr(), ops._stream(f1.device)),
                       "triad_similarity_matrix")
        return out


class TriadHotPath(TriadSimilarityMixin, torch.nn.Module):
    """Stand-alone module with just the state the hot path reads (model.py:348-351).  Used by
    bench.py / tests / smoke; a full model would mix TriadSimilarityMixin into MultiModalModel."""

    def __init__(self, temperature: float = 1.2, patch_sparsity_threshold: float = 0.3,
                 patch_sparsity_weight: float = 0.1):
        super().__init__()
        self.temperature = torch.nn.Parameter(torch.tensor(float(temperature)))
        self.patch_sparsity_threshold = patch_sparsity_threshold
        self.patch_sparsity_weight = patch_sparsity_weight

    def forward_features_av(self, audio_feats, visual_feats):
        clip, tok = self.compute_all_similarities_av(audio_feats, visual_feats)
        return self.compute_contrastive_loss_av(clip, tok)

    def forward_features_tv(self, text_feats, visual_feats, attention_mask):
        clip, tok = self.compute_all_similarities_tv(text_feats, visual_feats, attention_mask)
        return self.compute_contrastive_loss_tv(clip, tok)
