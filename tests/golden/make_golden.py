"""Generates tests/golden/*.pt by running the UNMODIFIED reference (via oracle/ref_shim.py) on seeded weights and
synthetic batches.  Needs a checkout of the reference (BEVBERT_REFERENCE); the tests only read the stored outputs:

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden.py [fixture ...]      # default: all of FIXTURES

Weights (synth.det_init_) and batches (synth.make_batch) are regenerated bit-identically from their seeds by
the tests, so only reference OUTPUTS are stored: per-item losses, logits, per-parameter gradient norms and a
few full gradients.  The reference has no tests or golden vectors of its own (SURVEY.md 4)."""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from bevbert_b200 import synth  # noqa: E402
from bevbert_b200.config import make_config  # noqa: E402
from bevbert_b200.model.pretrain_cmt import GlocalTextPathCMTPreTraining  # noqa: E402
from helpers import GOLDEN_THREADS, digest, golden_sample, small_config, small_synth  # noqa: E402

OUT_DIR = os.path.dirname(os.path.abspath(__file__))

FULL_GRADS = ["bert.embeddings.LayerNorm.weight", "bert.lang_encoder.layer.0.attention.self.query.bias",
              "bert.local_encoder.encoder.x_layers.0.visual_attention.att.query.bias",
              "bert.global_encoder.sprel_linear.weight", "bert.global_encoder.sprel_linear.bias",
              "bert.img_embeddings.loc_linear.weight", "bert.local_encoder.bev_pos_embeddings.0.weight"]

CASES = {
    "small_r2r": (lambda: small_config(), lambda: small_synth(), ["mlm", "sap", "masksem"]),
    "small_reverie": (lambda: small_config(obj_feat_size=768, obj_prob_size=100, pretrain_tasks=["mlm", "mrc", "sap", "og"]),
                      lambda: small_synth(obj_feat_size=768, obj_max=5, obj_prob_size=100), ["mlm", "mrc", "sap", "og"]),
    "config1_full_depth": (lambda: make_config(bev_dim=11, bev_res=1.0, hidden_dropout_prob=0.0,
                                               attention_probs_dropout_prob=0.0, feat_dropout=0.0),
                           lambda: small_synth(), ["mlm", "sap", "masksem"]),
}

# tests/test_oracle_vs_reference.py: weights / batch seeds and the edge-case inputs
RESTATEMENT_TASKS = ["mlm", "sap", "masksem"]
EDGE_CASES = {"longest_trajectory": lambda: small_synth(pano_min=21, pano_max=21),
              "empty_bev": lambda: small_synth(depth_zero_frac=1.0)}
BEV_SEEDS = (1, 2, 3)


def _ref_model(cfg, sd):
    from oracle import ref_shim
    ref = ref_shim.build_reference_model(cfg, sd).train()
    for m in ref.modules():
        if isinstance(m, torch.nn.Dropout):
            m.p = 0.0
        if isinstance(m, torch.nn.MultiheadAttention):
            m.dropout = 0.0
    return ref


def _seeded_sd(model_cls, cfg, seed):
    return {k: v.detach().clone() for k, v in synth.det_init_(model_cls(cfg), seed=seed).state_dict().items()}


def model_case(name):
    mk_cfg, mk_synth, tasks = CASES[name]
    cfg, scfg = mk_cfg(), mk_synth()
    sd = _seeded_sd(GlocalTextPathCMTPreTraining, cfg, 3)
    ref = _ref_model(cfg, sd)
    assert set(ref.state_dict().keys()) == set(sd.keys()), "state_dict key sets differ"
    for k, v in ref.state_dict().items():
        assert v.shape == sd[k].shape, k
    gold = {"state_dict_keys": sorted(sd.keys()), "shapes": {k: tuple(v.shape) for k, v in sd.items()}}
    for task in tasks:
        b = synth.make_batch(scfg, seed=7, task=task)
        ref.zero_grad()
        loss = ref(synth.clone_batch(b), task, compute_loss=True)
        loss.mean().backward()
        with torch.no_grad():
            logits = ref(synth.clone_batch(b), task, compute_loss=False)
        logits = logits if isinstance(logits, tuple) else (logits,)
        grads = {n: p.grad for n, p in ref.named_parameters() if p.grad is not None}
        gold[task] = {
            "loss": loss.detach().clone(),
            "logits": [t.detach().clone() for t in logits[:3]],
            "grad_norms": {n: float(g.norm()) for n, g in grads.items()},
            "grads": {n: grads[n].clone() for n in FULL_GRADS if n in grads},
        }
        print(name, task, "loss mean %.6f" % float(loss.mean()), "n_grads", len(grads))
    return gold


def oracle_vs_reference():
    """Per-item losses of the reference model on ragged-text and edge-case batches, and the reference BEV projector's
    cell index of every point, masks and pooled maps (tests/test_oracle_vs_reference.py)."""
    from oracle import bevbert_ref as R
    from oracle import ref_shim
    cfg = small_config()
    sd = _seeded_sd(GlocalTextPathCMTPreTraining, cfg, 5)
    ref = _ref_model(cfg, sd)
    gold = {"restatement": {}, "edge_cases": {}, "bev": {}}
    for task in RESTATEMENT_TASKS:
        b = synth.make_batch(small_synth(ragged_txt=True), seed=21, task=task)
        gold["restatement"][task] = ref(synth.clone_batch(b), task, compute_loss=True).detach().clone()
    for case, mk_synth in EDGE_CASES.items():
        gold["edge_cases"][case] = {}
        for task in ("sap", "mlm"):
            b = synth.make_batch(mk_synth(), seed=23, task=task)
            gold["edge_cases"][case][task] = ref(synth.clone_batch(b), task, compute_loss=True).detach().clone()
    _, pretrain_cmt = ref_shim.load_pretrain_modules(21, 0.5)
    projector, _ = pretrain_cmt.build_projector()
    bs = 4
    for seed in BEV_SEEDS:
        b = synth.make_batch(synth.SynthConfig(batch_size=bs), seed=seed)
        depths = (b["depths"] * 10).reshape(-1, 1, 14, 14)
        pc, mask = projector.forward(depths, b["T_c2w"].reshape(-1, 4, 4))
        pc = pc.reshape(bs, -1, 3) - b["S_w2c"]
        pc1 = torch.cat([pc, torch.ones(bs, pc.shape[1], 1)], -1) @ b["T_w2c"].squeeze(1).transpose(1, 2)
        bev, ob, sem, sem_mask = projector.project_bev(pc1[:, :, :3], mask.reshape(bs, -1), b["rgbs"].reshape(bs, -1, 768),
                                                       b["sems"].reshape(bs, -1, 40))
        # the cell of every reference point: project_bev computes it the same way (bev_utils.py:393-406) but does not
        # return it
        cell_idx = R.cell_index(pc1[:, :, :3], mask.reshape(bs, -1), 21, 0.5).to(torch.int16)
        gold["bev"][seed] = {"cell_idx": cell_idx, "bev_fts": digest(bev.reshape(bs, -1, 768)),
                             "bev_sems": digest(sem.reshape(bs, -1, 40)), "bev_sem_masks": sem_mask.reshape(bs, -1).clone(),
                             "bev_ob_masks": ob.reshape(bs, -1).clone()}
    return gold


def nav_reference():
    """GlocalTextPathNavCMT of the reference in its three modes (tests/test_nav_api_cpu.py)."""
    from oracle import ref_shim
    from bevbert_b200.model.nav_vilmodel import GlocalTextPathNavCMT
    from test_nav_api_cpu import nav_batches, nav_config
    cfg = nav_config()
    sd = _seeded_sd(GlocalTextPathNavCMT, cfg, 4)
    ref = ref_shim.load_nav_module().GlocalTextPathNavCMT(cfg)
    ref.load_state_dict(sd)
    ref.eval()
    lang, pano, nav = nav_batches()
    with torch.no_grad():
        t = ref("language", lang)
        pe, pm = ref("panorama", pano)
        nav["txt_embeds"] = t
        out = ref("navigation", nav)
    return {"state_dict_keys": sorted(ref.state_dict().keys()), "language": golden_sample(t),
            "panorama": (golden_sample(pe), pm.clone()),
            "navigation": dict({k: out[k].clone() for k in ("global_logits", "local_logits", "fused_logits")},
                               gmap_embeds=golden_sample(out["gmap_embeds"]))}


def adamw_reference():
    """Parameters after the steps of tests/test_optim_cpu.py through the reference AdamW (pretrain_src/optim/adamw.py)
    with torch's grad-norm clip."""
    import importlib.util
    from oracle import ref_shim
    from test_optim_cpu import ADAMW_STEPS, _params, step_grads
    spec = importlib.util.spec_from_file_location("_ref_adamw", os.path.join(ref_shim.REF_ROOT, "pretrain_src", "optim",
                                                                             "adamw.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    a = _params()
    opt = mod.AdamW([{"params": [a[0], a[2], a[3]], "weight_decay": 0.01}, {"params": [a[1]], "weight_decay": 0.0}],
                       lr=3e-3, betas=(0.9, 0.98))
    g = torch.Generator().manual_seed(2)
    for step in range(ADAMW_STEPS):
        for p, gr in zip(a, step_grads(a, step, g)):
            p.grad = gr
        torch.nn.utils.clip_grad_norm_(a, 5.0)
        opt.step()
    return {"params": [p.detach().clone() for p in a]}


FIXTURES = dict({name: (lambda name=name: model_case(name)) for name in CASES},
                oracle_vs_reference=oracle_vs_reference, nav_reference=nav_reference, adamw_reference=adamw_reference)


def main(names):
    torch.set_num_threads(GOLDEN_THREADS)
    for name in names or FIXTURES:
        torch.save(FIXTURES[name](), os.path.join(OUT_DIR, name + ".pt"))


if __name__ == "__main__":
    main(sys.argv[1:])
