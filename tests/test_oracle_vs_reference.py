"""Pins the oracle to the real reference: the unmodified reference modules ran on the same weights and batches as the
restatement, and their outputs are stored in tests/golden/oracle_vs_reference.pt (written by
tests/golden/make_golden.py through oracle/ref_shim.py)."""
import os
import sys

import pytest
import torch

from bevbert_b200 import synth
from bevbert_b200.model.pretrain_cmt import GlocalTextPathCMTPreTraining
from helpers import digest, golden_threads, small_config, small_synth
from oracle import bevbert_ref as R

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
sys.path.insert(0, GOLD)
import make_golden  # noqa: E402

REF = torch.load(os.path.join(GOLD, "oracle_vs_reference.pt"), weights_only=True)


@pytest.fixture(autouse=True)
def _golden_threads():
    with golden_threads():
        yield


def _seeded_sd(cfg):
    return {k: v.detach().clone() for k, v in synth.det_init_(GlocalTextPathCMTPreTraining(cfg), seed=5).state_dict().items()}


@pytest.mark.parametrize("task", ["mlm", "sap", "masksem"])
def test_restatement_equals_reference(task):
    cfg, scfg = small_config(), small_synth(ragged_txt=True)
    sd = _seeded_sd(cfg)
    b = synth.make_batch(scfg, seed=21, task=task)
    want = REF["restatement"][task]
    got = R.forward(sd, synth.clone_batch(b), task, R.OracleConfig(cfg))
    assert torch.allclose(got, want, rtol=1e-5, atol=1e-6), float((got - want).abs().max())


@pytest.mark.parametrize("case", ["longest_trajectory", "empty_bev"])
def test_restatement_equals_reference_on_edge_cases(case):
    """SURVEY section 4 property cases, pinned on the unmodified reference: 21 panoramas per trajectory (TRAIN_MAX_STEP + 1,
    dataset.py:185-187) and depth maps that are all zero (every point dropped, all BEV cells empty)."""
    cfg = small_config()
    scfg = make_golden.EDGE_CASES[case]()
    sd = _seeded_sd(cfg)
    for task in ("sap", "mlm"):
        b = synth.make_batch(scfg, seed=23, task=task)
        want = REF["edge_cases"][case][task]
        got = R.forward(sd, synth.clone_batch(b), task, R.OracleConfig(cfg))
        assert torch.isfinite(want).all()
        assert torch.allclose(got, want, rtol=1e-5, atol=1e-6), (task, float((got - want).abs().max()))


def test_bev_projection_matches_reference_bit_for_bit():
    """lift + project_bev of the reference (torch bmm / matmul + scatter_mean stub) vs the fixed-order oracle:
    cell indices, pooled features, semantic maps and masks.  The reference's pooled feature and semantic maps are
    stored as SHA-256 digests of their bytes."""
    mismatched = 0
    total = 0
    for seed in make_golden.BEV_SEEDS:
        ref = REF["bev"][seed]
        b = synth.make_batch(synth.SynthConfig(batch_size=4), seed=seed)
        ob_ = dict(b)
        R.lift_splat(ob_, 21, 0.5)
        same = digest(ob_["bev_fts"]) == ref["bev_fts"]
        # the reference leaves the order of the 4-term dot products to bmm/matmul; count index flips instead of failing
        ref_idx = ref["cell_idx"].long()
        mismatched += int((ref_idx != ob_["bev_cell_idx"]).sum())
        total += ref_idx.numel()
        if same:
            assert digest(ob_["bev_sems"]) == ref["bev_sems"]
            assert torch.equal(ob_["bev_sem_masks"], ref["bev_sem_masks"])
            assert torch.equal(ob_["bev_ob_masks"], ref["bev_ob_masks"])
    assert mismatched <= total * 1e-5, "cell-index disagreement with the reference: %d of %d" % (mismatched, total)
