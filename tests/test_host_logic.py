"""CPU tier: host-side logic that needs no GPU — the lazy statistics mapping, the top-k merge order of the
gallery-sharded retrieval, the staged-reference recipe (oracle/build_ref.py), and bench.py's CPU arm wiring."""
import copy
import hashlib
import json
import os
import pickle
import shutil

import pytest
import torch

from oracle import oracle as O


def test_lazy_stats_is_a_mapping_with_the_reference_keys():
    from triad_b200.model import LazyStats
    clip = torch.randn(6, 6, dtype=torch.float64)
    B = 6
    d = torch.diagonal(clip)
    off = clip[~torch.eye(B, dtype=torch.bool)]
    sums = torch.tensor([0.0, d.sum(), (d * d).sum(), off.sum(), (off * off).sum(), off.max(), 0.0, 0.0], dtype=torch.float64)
    stats = LazyStats(sums, B, "av")
    want = O.similarity_stats(clip, "av")
    assert sorted(stats.keys()) == sorted(want) and len(stats) == 6
    for k, v in want.items():
        assert k in stats and abs(stats[k] - v) < 1e-9
    d2 = {}
    d2.update(stats)                                   # train.py:1080 (wandb_dict.update)
    assert d2 == stats.to_dict() == {**stats} == dict(stats)
    assert json.loads(json.dumps(stats.to_dict())) == pytest.approx(d2)
    assert pickle.loads(pickle.dumps(stats)) == d2 and copy.deepcopy(stats) == d2
    with pytest.raises(TypeError):
        json.dumps(stats)                              # loud, not a silent '{}' (it is not a dict subclass)


def test_merge_topk_order():
    from triad_b200.dist import merge_topk
    s = torch.tensor([1.0, 3.0, 3.0, 2.0, 3.0, float("-inf")])
    i = torch.tensor([9, 7, 2, 5, 4, torch.iinfo(torch.int64).max])
    ms, mi = merge_topk(s, i, 4)
    assert mi.tolist() == [2, 4, 7, 5] and ms.tolist() == [3.0, 3.0, 3.0, 2.0]   # score desc, ties to the lower id


# SHA-256 of the reference's src/model.py and src/retrieval.py, taken from the reference tree when oracle/_ref/ was staged
REFERENCE_SHA256 = {
    "model.py": "5d5d00fccac98ce98fe474ff25569cc2f5b715776cfb7b5850f275d9a1b5eafc",
    "retrieval.py": "9029727c6c9729adf8f5dbace7fa95a0e69de17f26ea401c89ff19c2dc8871a2",
}


def test_staged_reference_is_the_reference_byte_for_byte(tmp_path, monkeypatch):
    from oracle import build_ref, ref_loader
    for name, digest in REFERENCE_SHA256.items():
        with open(os.path.join(build_ref.OUT, name), "rb") as f:
            assert hashlib.sha256(f.read()).hexdigest() == digest, name
    # the staging recipe, run on a reference tree laid out like the original: byte-for-byte copies, and the manifest
    # that is kept in oracle/_ref/
    src_root = tmp_path / "reference"
    for rel in build_ref.FILES:
        (src_root / rel).parent.mkdir(parents=True, exist_ok=True)
        shutil.copyfile(os.path.join(build_ref.OUT, os.path.basename(rel)), src_root / rel)
    staged = tmp_path / "staged"
    monkeypatch.setattr(build_ref, "REF_ROOT", str(src_root))
    monkeypatch.setattr(build_ref, "OUT", str(staged))
    assert build_ref.build()
    with open(staged / "MANIFEST.json") as f, open(os.path.join(ref_loader.REF_DIR, "MANIFEST.json")) as g:
        assert json.load(f) == json.load(g)
    for rel in build_ref.FILES:
        assert (staged / os.path.basename(rel)).read_bytes() == (src_root / rel).read_bytes()
    ref = ref_loader.load()
    assert ref is not None and hasattr(ref[0], "MultiModalModel") and hasattr(ref[1], "compute_recall_at_k")


def test_reference_arm_runs_the_staged_reference_and_matches_the_oracle():
    """bench.py's CPU arm: one step of the reference's own methods (regularisers bound to zero) equals the oracle's
    contrastive-only closed form on the same inputs — value and gradients."""
    from oracle import ref_loader
    ref = ref_loader.load()
    if ref is None:
        pytest.skip("oracle/_ref not staged")
    M = ref[0].MultiModalModel
    for masked in (False, True):
        q, v, mask = O.make_inputs(4, 9, 20, 16, torch.float32, seed=2, masked=masked, min_len=2)
        stub = ref_loader.make_stub(M, 1.5, regularizers=False)
        q.requires_grad_(True); v.requires_grad_(True)
        if mask is None:
            clip, tok = M.compute_all_similarities_av(stub, q, v)
            total, con = M.compute_contrastive_loss_av(stub, clip, tok)[:2]
        else:
            clip, tok = M.compute_all_similarities_tv(stub, q, v, mask)
            total = con = M.compute_contrastive_loss_tv(stub, clip, tok)[0]
        total.backward()
        want = O.contrastive_step_closed_form(q.detach(), v.detach(), 1.5, mask)
        assert abs(total.item() - con.item()) < 1e-7 and abs(con.item() - want["loss"].item()) < 1e-5
        assert torch.allclose(q.grad.double(), want["dq"], atol=1e-6) and torch.allclose(v.grad.double(), want["dv"], atol=1e-6)
        assert abs(stub.temperature.grad.item() - want["dT"].item()) < 1e-5


def test_bench_cpu_arm_reports_reference_kind():
    import bench
    step, kind, what = bench.cpu_reference_step_factory(dict(Nq=5, Nv=8, D=16, masked=False), 3)
    from oracle import ref_loader
    assert kind == ("reference" if ref_loader.available() else "port")
    assert step() == step()                               # deterministic, finite


def test_chunk_budget_queries_the_driver_once_per_ttl(monkeypatch):
    """regularizers.chunk_budget caps a chunk of N at a quarter of the free memory; the driver query behind it
    (cudaMemGetInfo: milliseconds, more while NVML clients talk to the driver) is cached, not issued per training step."""
    from triad_b200 import regularizers as R
    calls = []

    def fake_mem_get_info(device=None):
        calls.append(device)
        return (40 << 30, 180 << 30)

    monkeypatch.setattr(torch.cuda, "mem_get_info", fake_mem_get_info)
    monkeypatch.setattr(torch.cuda, "current_device", lambda: 0)
    R._free_cache.clear()
    assert R.chunk_budget("cuda:0", 16 << 30) == 10 << 30        # free // 4
    assert R.chunk_budget("cuda:0", 16 << 30) == 10 << 30
    assert R.chunk_budget("cuda:0", 4 << 30) == 4 << 30          # the caller's bound when it is the smaller one
    assert len(calls) == 1
    assert R.chunk_budget("cuda:0", 4096) == 4096 and len(calls) == 1      # test-sized chunks never ask
    monkeypatch.setattr(R, "FREE_MEMORY_TTL_S", -1.0)            # expired: asks again
    R.chunk_budget("cuda:0", 16 << 30)
    assert len(calls) == 2
    R._free_cache.clear()


def test_clock_sampler_degrades_without_a_gpu():
    """bench.ClockSampler never raises: no NVML / no nvidia-smi gives an empty summary (the bench line still prints)."""
    import bench
    import time as _t
    with bench.ClockSampler(0) as c:
        _t.sleep(0.03)
    s = c.summary()
    assert set(s) >= {"sm_mhz", "sm_max_mhz", "reasons", "samples"}
    if s["samples"] == 0:
        assert s["sm_mhz"] is None and s["reasons"] == []
