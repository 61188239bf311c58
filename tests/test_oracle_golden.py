"""The CPU oracle (oracle/bevbert_ref.py) against golden outputs of the unmodified reference
(tests/golden/*.pt, produced by tests/golden/make_golden.py in the build container)."""
import os

import pytest
import torch

from bevbert_b200 import synth
from bevbert_b200.model.pretrain_cmt import GlocalTextPathCMTPreTraining
from helpers import golden_threads
from oracle import bevbert_ref as R

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(autouse=True)
def _golden_threads():
    with golden_threads():
        yield


def _cases():
    import sys
    sys.path.insert(0, GOLD)
    import make_golden
    return make_golden.CASES


@pytest.mark.parametrize("name", ["small_r2r", "small_reverie"])
def test_oracle_reproduces_reference_outputs(name):
    mk_cfg, mk_synth, tasks = _cases()[name]
    cfg, scfg = mk_cfg(), mk_synth()
    gold = torch.load(os.path.join(GOLD, name + ".pt"), weights_only=False)
    model = synth.det_init_(GlocalTextPathCMTPreTraining(cfg), seed=3)
    # drop-in surface: identical state_dict keys and shapes
    assert sorted(model.state_dict().keys()) == gold["state_dict_keys"]
    assert {k: tuple(v.shape) for k, v in model.state_dict().items()} == gold["shapes"]
    sd = {k: v.detach().clone().requires_grad_(True) for k, v in model.state_dict().items()}
    ocfg = R.OracleConfig(cfg)
    for task in tasks:
        b = synth.make_batch(scfg, seed=7, task=task)
        for v in sd.values():
            v.grad = None
        loss = R.forward(sd, synth.clone_batch(b), task, ocfg)
        loss.mean().backward()
        g = gold[task]
        assert torch.allclose(loss, g["loss"], rtol=1e-5, atol=1e-6), task
        logits = R.forward({k: v.detach() for k, v in sd.items()}, synth.clone_batch(b), task, ocfg, compute_loss=False)
        logits = logits if isinstance(logits, tuple) else (logits,)
        for a, r in zip(logits[:3], g["logits"]):
            fin = torch.isfinite(r)
            assert torch.equal(torch.isfinite(a), fin)
            assert torch.allclose(a[fin], r[fin], rtol=1e-4, atol=1e-5)
        top = max(g["grad_norms"].values())
        for n, gn in g["grad_norms"].items():
            assert sd[n].grad is not None, n
            assert abs(float(sd[n].grad.norm()) - gn) <= 1e-3 * max(gn, 1e-4 * top), (task, n)
        for n, gr in g["grads"].items():
            assert torch.allclose(sd[n].grad, gr, rtol=1e-3, atol=1e-4 * float(gr.abs().max()) + 1e-9), (task, n)
