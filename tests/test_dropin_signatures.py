"""CPU tier: the drop-in surface keeps the reference's names, positional parameters and MRO behaviour
(SURVEY.md §8(b)): the frozen copy of the expected signatures below is checked against the drop-in and against the
reference's own source (the staged copy in oracle/_ref/)."""
import inspect

import pytest
import torch

import triad_b200
from triad_b200 import retrieval as R
from triad_b200.model import TriadSimilarityMixin

# (name, positional parameters after self) — src/model.py:355-368, :370-392, :430-472, :490-514, :544-593
MODEL_METHODS = {
    "compute_similarity_matrix": ["feats1", "feats2"],
    "compute_all_similarities_av": ["audio_feats", "visual_feats"],
    "compute_all_similarities_tv": ["text_feats", "visual_feats", "attention_mask"],
    "compute_contrastive_loss_av": ["clip_sims", "token_sims"],
    "compute_contrastive_loss_tv": ["clip_sims", "token_sims"],
    "compute_regularization_losses_av": ["token_sims"],
    "compute_regularization_losses_tv": ["token_sims"],
}
# src/retrieval.py:106-115, :117-144, :146, :190-198, :250
RETRIEVAL_FUNCS = {
    "aggregator_av_a2v": ["a_feats", "v_feats", "temperature"],
    "aggregator_av_v2a": ["a_feats", "v_feats", "temperature"],
    "aggregator_tv_t2v": ["t_feats", "v_feats", "temperature"],
    "aggregator_tv_v2t": ["t_feats", "v_feats", "temperature"],
    "compute_recall_at_k": ["sim_matrix"],
    "compute_av_retrieval_metrics": ["model", "dataset", "subset_file", "device"],
    "compute_tv_retrieval_metrics": ["model", "dataset", "subset_file", "device"],
}


def _params(fn, skip_self):
    names = list(inspect.signature(fn).parameters)
    return names[1:] if skip_self else names


def test_mixin_keeps_the_reference_method_surface():
    for name, params in MODEL_METHODS.items():
        assert _params(getattr(TriadSimilarityMixin, name), True) == params, name
    for name, params in RETRIEVAL_FUNCS.items():
        assert _params(getattr(R, name), False) == params, name


def test_mixin_shadows_the_host_class_methods():
    """class MultiModalModel(TriadSimilarityMixin, nn.Module): the mixin's methods win (INTEGRATION.md §3)."""
    class Host(torch.nn.Module):
        def compute_all_similarities_av(self, audio_feats, visual_feats):
            return "reference"

        def forward_audio_visual(self, a, v):                     # model.py:487-488 calls the methods by name
            return self.compute_all_similarities_av(a, v)

    class Patched(TriadSimilarityMixin, Host):
        pass

    assert Patched.compute_all_similarities_av is TriadSimilarityMixin.compute_all_similarities_av
    m = Patched()
    m.temperature = torch.nn.Parameter(torch.tensor(1.2))
    with pytest.raises(RuntimeError):                             # reaches the CUDA-only path: no silent fallback
        m.forward_audio_visual(torch.randn(2, 3, 64), torch.randn(2, 5, 64))


def test_signatures_match_the_reference_source():
    from oracle import ref_loader
    ref = ref_loader.load()
    assert ref is not None, "oracle/_ref/ holds no staged reference"
    ref_model, ref_retrieval = ref
    M = ref_model.MultiModalModel
    for name, params in MODEL_METHODS.items():
        assert _params(getattr(M, name), True) == params, name
    for name, params in RETRIEVAL_FUNCS.items():
        assert _params(getattr(ref_retrieval, name), False) == params, name
    # defaults the drop-in module mirrors (model.py:331-341)
    ref_defaults = {k: v.default for k, v in inspect.signature(M.__init__).parameters.items()}
    mine = {k: v.default for k, v in inspect.signature(triad_b200.TriadHotPath.__init__).parameters.items()}
    for k in ("temperature", "patch_sparsity_threshold", "patch_sparsity_weight"):
        assert mine[k] == ref_defaults[k], k
