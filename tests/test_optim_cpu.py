"""oracle/adamw_ref.py (the checker of the CUDA optimizer kernel) is pinned to the UNMODIFIED reference optimizer
(pretrain_src/optim/adamw.py) + torch's clip_grad_norm_ on CPU, through the parameters the reference reached on the same
gradients (tests/golden/adamw_reference.pt, written by tests/golden/make_golden.py); the kernel itself is tested in
tests/test_optim_gpu.py against that restatement."""
import os

import torch

from oracle import adamw_ref

ADAMW_STEPS = 9
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "adamw_reference.pt")


def _params(seed=1):
    g = torch.Generator().manual_seed(seed)
    return [torch.nn.Parameter(torch.randn(s, generator=g)) for s in ((7, 5), (11,), (3, 3), (130, 9))]


def step_grads(params, step, g):
    """The gradients of one step: a 10x larger step 4, and one parameter without a gradient per step."""
    grads = [torch.randn(p.shape, generator=g) * (10.0 if step == 4 else 1.0) for p in params]
    skip = step % 4
    return [None if i == skip else gr for i, gr in enumerate(grads)]


def test_oracle_adamw_matches_reference_optimizer():
    b = _params()
    wds = [0.01, 0.0, 0.01, 0.01]
    mine = adamw_ref.AdamWRef([p.data for p in b], lr=3e-3, betas=(0.9, 0.98), eps=1e-6, weight_decay=wds)
    g = torch.Generator().manual_seed(2)
    for step in range(ADAMW_STEPS):
        mg = step_grads(b, step, g)
        a = [torch.nn.Parameter(p.detach().clone()) for p in b]
        for p, gr in zip(a, mg):
            p.grad = None if gr is None else gr.clone()
        n_ref = torch.nn.utils.clip_grad_norm_(a, 5.0)
        n_mine = adamw_ref.clip_grad_norm_([x for x in mg if x is not None], 5.0)
        assert abs(float(n_ref) - float(n_mine)) <= 1e-5 * float(n_ref)
        mine.step(mg)
    want = torch.load(GOLD, weights_only=True)["params"]
    for pa, pb in zip(want, b):
        assert torch.allclose(pa, pb.detach(), rtol=1e-6, atol=1e-7)


def test_param_groups_follow_reference_no_decay_rule():
    from bevbert_b200.optim import build_param_groups
    m = torch.nn.Module()
    m.dense = torch.nn.Linear(4, 4)
    m.LayerNorm = torch.nn.LayerNorm(4)
    groups = build_param_groups(m, 0.01)
    assert [tuple(p.shape) for p in groups[0]["params"]] == [(4, 4)] and groups[0]["weight_decay"] == 0.01
    assert len(groups[1]["params"]) == 3 and groups[1]["weight_decay"] == 0.0
