"""Shared helpers for the parity tests."""
import contextlib
import hashlib

import torch

from bevbert_b200 import synth
from bevbert_b200.config import make_config

# tests/golden/make_golden.py runs the reference with this many intra-op threads.  torch splits fp32 reductions on the
# CPU by thread count, so the oracle reproduces the stored outputs bit for bit only with the same count.
GOLDEN_THREADS = 8


@contextlib.contextmanager
def golden_threads():
    prev = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    try:
        yield
    finally:
        torch.set_num_threads(prev)


def golden_sample(t, n=8192):
    """n elements of `t` at fixed positions (synth's reproducible generator): what tests/golden/ keeps of an output too
    large to store whole."""
    flat = t.detach().reshape(-1)
    return flat[synth.det_randint((n,), 0, 0, 0, flat.numel() - 1)].clone()


def digest(t):
    """SHA-256 of a tensor's dtype, shape and bytes: a bit-exact comparison with an output too large to store."""
    t = t.detach().contiguous()
    h = hashlib.sha256(("%s %s " % (t.dtype, tuple(t.shape))).encode())
    h.update(t.view(torch.uint8).reshape(-1).numpy().tobytes())
    return h.hexdigest()


SMALL = dict(num_l_layers=2, num_x_layers=2, num_pano_layers=1, vocab_size=3000, bev_dim=11, bev_res=1.0,
             hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0, feat_dropout=0.0)


def small_config(**kw):
    d = dict(SMALL)
    d.update(kw)
    return make_config(**d)


def small_synth(**kw):
    d = dict(batch_size=2, bev_dim=11, bev_res=1.0, pano_min=4, pano_max=6, gmap_min=8, gmap_max=8, vocab_hi=2000)
    d.update(kw)
    return synth.SynthConfig(**d)


def rel_l2(a, b):
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))


def grad_report(named_grads, ref_grads, floor_frac=1e-4):
    """max over parameters of ||g - g_ref|| / max(||g_ref||, floor) where floor = floor_frac * largest
    reference-gradient norm (gradients that are mathematically zero -- e.g. the key bias -- are noise)."""
    top = max(float(g.norm()) for g in ref_grads.values() if g is not None)
    worst, worst_name = 0.0, None
    for n, g in named_grads.items():
        r = ref_grads.get(n)
        if r is None and g is None:
            continue
        assert r is not None and g is not None, "gradient presence differs for %s" % n
        e = float((g.detach().float().cpu() - r.detach().float().cpu()).norm()) / max(float(r.norm()), floor_frac * top)
        if e > worst:
            worst, worst_name = e, n
    return worst, worst_name


def grad_errors(named_grads, ref_grads, floor_frac=1e-2):
    """per-parameter relative errors (same definition as grad_report) + the global relative L2 error over all
    gradients concatenated."""
    top = max(float(g.norm()) for g in ref_grads.values() if g is not None)
    errs, num, den = {}, 0.0, 0.0
    for n, g in named_grads.items():
        r = ref_grads.get(n)
        if r is None and g is None:
            continue
        assert r is not None and g is not None, "gradient presence differs for %s" % n
        d = float((g.detach().float().cpu() - r.detach().float().cpu()).norm())
        errs[n] = d / max(float(r.norm()), floor_frac * top)
        num += d * d
        den += float(r.norm()) ** 2
    return errs, (num / max(den, 1e-60)) ** 0.5
