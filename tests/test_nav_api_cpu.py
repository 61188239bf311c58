"""Agent-side per-step API (GlocalTextPathNavCMT.forward(mode, batch), map_nav_src/models/vilmodel.py:889-912):
host logic on CPU with emulated kernels vs the oracle, and the oracle vs the unmodified reference."""
import os

import torch

from bevbert_b200 import synth
from bevbert_b200.model.nav_vilmodel import GlocalTextPathNavCMT
from helpers import golden_sample, golden_threads, small_config, small_synth
from oracle import bevbert_ref as R


def nav_config(**kw):
    return small_config(fix_lang_embedding=False, fix_pano_embedding=False, fix_local_branch=False, **kw)


def nav_batches(B=3, G=7, K=4, D=11, seed=3, H=768, obj=0):
    """language / panorama / navigation inputs shaped like map_nav_src/r2r/agent.py:_nav_*_variable."""
    u = lambda shape, s, lo=-1.0, hi=1.0: synth.det_uniform(shape, seed, s, lo, hi)
    L = 30
    txt_ids = synth.det_randint((B, L), seed, 1, 1000, 1999)
    txt_lens = torch.tensor([L, L - 7, L - 11][:B])
    txt_masks = torch.arange(L)[None] < txt_lens[:, None]
    lang = {"txt_ids": txt_ids * txt_masks, "txt_masks": txt_masks}
    V = 36
    view_lens = torch.full((B,), V)
    obj_lens = torch.tensor([obj, max(obj - 2, 0), 0][:B]) if obj else None
    Vt = V + (int(obj_lens.max()) if obj else 0)
    pano = {"view_img_fts": u((B, V, H), 2, -1.7, 1.7), "obj_img_fts": u((B, max(obj, 1), H), 3) if obj else None,
            "loc_fts": u((B, Vt, 7), 4), "nav_types": synth.det_randint((B, Vt), seed, 5, 0, 1), "view_lens": view_lens,
            "obj_lens": obj_lens}
    gmap_lens = torch.tensor([G, G - 2, G - 3][:B])
    gmask = torch.arange(G)[None] < gmap_lens[:, None]
    vpids = [[None] + ["s%dn%d" % (i, j) for j in range(1, int(gmap_lens[i]))] for i in range(B)]
    visited = torch.zeros(B, G, dtype=torch.bool)
    visited[:, 1:3] = True
    cand_vpids = [[None, vpids[i][1], vpids[i][3], vpids[i][-1]][:K] for i in range(B)]
    n = D * D
    cand_idx = torch.tensor([[(n - 1) // 2, 5 + i, 17 + i, 40 + i][:K] for i in range(B)])
    navm = torch.zeros(B, n, dtype=torch.bool)
    navm[torch.arange(B)[:, None], cand_idx] = True
    pd = u((B, G, G), 6, 0.0, 1.0)
    pd = (pd + pd.transpose(1, 2)) * gmask[:, :, None] * gmask[:, None, :]
    nav = {"txt_masks": txt_masks, "gmap_img_embeds": u((B, G, H), 7) * gmask[:, :, None], "gmap_step_ids": synth.det_randint((B, G), seed, 8, 0, 5) * gmask,
           "gmap_pos_fts": u((B, G, 7), 9), "gmap_masks": gmask, "gmap_pair_dists": pd, "gmap_visited_masks": visited,
           "gmap_vpids": vpids, "bev_fts": u((B, n, H), 10, -1.7, 1.7), "bev_pos_fts": u((B, n, 10), 11),
           "bev_masks": torch.ones(B, n, dtype=torch.bool), "bev_nav_masks": navm, "bev_cand_idxs": cand_idx,
           "bev_cand_vpids": cand_vpids, "obj_embeds": None, "obj_masks": None}
    return lang, pano, nav


def _check_outs(a, r, tol=1e-4):
    for k in ("gmap_embeds", "global_logits", "local_logits", "fused_logits"):
        fin = torch.isfinite(r[k])
        assert torch.equal(torch.isfinite(a[k]), fin), k
        assert torch.allclose(a[k][fin], r[k][fin], rtol=tol, atol=tol), (k, float((a[k][fin] - r[k][fin]).abs().max()))


def test_nav_modes_match_oracle(emu):
    cfg = nav_config()
    model = synth.det_init_(GlocalTextPathNavCMT(cfg), seed=4).train()
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    ocfg = R.OracleConfig(cfg)
    lang, pano, nav = nav_batches()
    t = model("language", lang)
    rt_ = R.nav_forward(sd, "language", lang, ocfg)
    assert torch.allclose(t, rt_, rtol=1e-4, atol=1e-5)
    pe, pm = model("panorama", pano)
    rpe, rpm = R.nav_forward(sd, "panorama", pano, ocfg)
    assert torch.equal(pm, rpm) and torch.allclose(pe, rpe, rtol=1e-4, atol=1e-5)
    nav["txt_embeds"] = rt_
    out = model("navigation", nav)
    ref = R.nav_forward(sd, "navigation", nav, ocfg)
    _check_outs(out, ref)
    # gradients flow back to the fp32 API inputs and the parameters
    te = rt_.clone().requires_grad_(True)
    nav["txt_embeds"] = te
    o = model("navigation", nav)
    o["fused_logits"][torch.isfinite(o["fused_logits"])].sum().backward()
    assert te.grad is not None and float(te.grad.abs().sum()) > 0
    assert model.global_sap_head.net[0].weight.grad is not None


def test_nav_oracle_equals_reference():
    """The oracle against the unmodified reference class on the same weights and inputs (its outputs, the large ones
    at fixed sample positions, stored in tests/golden/nav_reference.pt by tests/golden/make_golden.py)."""
    cfg = nav_config()
    ours = synth.det_init_(GlocalTextPathNavCMT(cfg), seed=4)
    sd = {k: v.detach().clone() for k, v in ours.state_dict().items()}
    ref = torch.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "nav_reference.pt"),
                     weights_only=True)
    assert set(ref["state_dict_keys"]) == set(sd.keys())
    ocfg = R.OracleConfig(cfg)
    lang, pano, nav = nav_batches()
    with torch.no_grad(), golden_threads():
        t = R.nav_forward(sd, "language", lang, ocfg)
        assert torch.allclose(golden_sample(t), ref["language"], rtol=1e-5, atol=1e-6)
        pe, pm = ref["panorama"]
        ope, opm = R.nav_forward(sd, "panorama", pano, ocfg)
        assert torch.equal(pm, opm) and torch.allclose(golden_sample(ope), pe, rtol=1e-5, atol=1e-6)
        nav["txt_embeds"] = t
        want = ref["navigation"]
        got = R.nav_forward(sd, "navigation", nav, ocfg)
    _check_outs(dict(got, gmap_embeds=golden_sample(got["gmap_embeds"])), want, tol=1e-5)
