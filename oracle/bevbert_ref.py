"""TEST INFRASTRUCTURE ONLY -- CPU/fp32 oracle for the BEVBert hybrid-map encoder hot path.

A plain-PyTorch *functional* restatement of the reference's algorithm, evaluated over a flat
``state_dict`` (same keys as the reference model) so that any set of weights can be checked.  It exists to
(a) check the CUDA path in tests/, __graft_entry__.smoke() and (b) serve as the timed CPU baseline
in bench.py (`cpu_baseline`, `--impl reference`), because the reference itself (/root/reference) cannot
travel to the GPU box.  The product package never imports it.

Pinned against the real reference: tests/golden/make_golden.py runs the unmodified reference modules
(oracle/ref_shim.py) on seeded weights/batches and stores their outputs in tests/golden/*.pt, which
tests/test_oracle_golden.py and tests/test_oracle_vs_reference.py compare with.  The reference ships
no tests or golden vectors of its own (SURVEY.md 4, 8c).

Every function cites the reference lines it restates (paths relative to the reference root,
pretrain_src/model/...).  Dropout is taken as p = 0 unless `drop_p` is given (parity runs use 0).
"""
import math
from collections import defaultdict

import torch
import torch.nn.functional as F

NEG = -10000.0


# ----------------------------------------------------------------------------- small helpers
def _lin(sd, p, x):
    return F.linear(x, sd[p + ".weight"], sd.get(p + ".bias"))


def _ln(sd, p, x, eps):
    return F.layer_norm(x, (x.shape[-1],), sd[p + ".weight"], sd[p + ".bias"], eps)


def _gelu(x):  # vilmodel.py:31-37
    return x * 0.5 * (1.0 + torch.erf(x / math.sqrt(2.0)))


def seq_mask(lens, max_len=None):  # ops.py:36-44
    max_len = int(max(lens)) if max_len is None else max_len
    return torch.arange(max_len, device=lens.device)[None, :] < lens[:, None]


def neg_mask(mask):  # ops.py:25-34  (N,L) -> (N,1,1,L) additive -10000
    return (1.0 - mask[:, None, None, :].to(torch.float32)) * NEG


def _drop(x, p):
    return F.dropout(x, p, training=True) if p > 0 else x


def _heads(x, nh):
    n, l, d = x.shape
    return x.view(n, l, nh, d // nh).permute(0, 2, 1, 3)


# ----------------------------------------------------------------------------- BERT blocks
def attention_core(q, k, v, add_mask, nh, p=0.0):
    """vilmodel.py:112-137 / 330-351: softmax(QK^T/sqrt(d) + mask) V with merged heads."""
    q, k, v = _heads(q, nh), _heads(k, nh), _heads(v, nh)
    s = torch.matmul(q, k.transpose(-1, -2)) / math.sqrt(q.shape[-1])
    if add_mask is not None:
        s = s + add_mask
    pr = _drop(torch.softmax(s, dim=-1), p)
    ctx = torch.matmul(pr, v).permute(0, 2, 1, 3).contiguous()
    return ctx.view(ctx.shape[0], ctx.shape[1], -1)


def self_output(sd, p, h, inp, eps, dp):  # BertSelfOutput / BertOutput, vilmodel.py:150-154,189-193
    return _ln(sd, p + ".LayerNorm", _drop(_lin(sd, p + ".dense", h), dp) + inp, eps)


def bert_attention(sd, p, x, add_mask, cfg):  # vilmodel.py:156-166
    ctx = attention_core(_lin(sd, p + ".self.query", x), _lin(sd, p + ".self.key", x),
                         _lin(sd, p + ".self.value", x), add_mask, cfg.num_attention_heads, cfg.drop_p)
    return self_output(sd, p + ".output", ctx, x, cfg.layer_norm_eps, cfg.drop_p)


def ffn(sd, p_inter, p_out, x, cfg):  # vilmodel.py:168-193
    return self_output(sd, p_out, _gelu(_lin(sd, p_inter + ".dense", x)), x, cfg.layer_norm_eps, cfg.drop_p)


def bert_layer(sd, p, x, add_mask, cfg):  # vilmodel.py:195-208
    a = bert_attention(sd, p + ".attention", x, add_mask, cfg)
    return ffn(sd, p + ".intermediate", p + ".output", a, cfg)


def cross_attention(sd, p, x, ctx, ctx_mask, cfg):  # BertXAttention, vilmodel.py:354-363 (+301-352)
    c = attention_core(_lin(sd, p + ".att.query", x), _lin(sd, p + ".att.key", ctx), _lin(sd, p + ".att.value", ctx),
                       ctx_mask, cfg.num_attention_heads, cfg.drop_p)
    return self_output(sd, p + ".output", c, x, cfg.layer_norm_eps, cfg.drop_p)


def xlayer_visn(sd, p, lang, lang_mask, visn, visn_mask, sprels, cfg):  # GraphLXRTXLayer.forward, :383-398
    v = cross_attention(sd, p + ".visual_attention", visn, lang, lang_mask, cfg)
    m = visn_mask + sprels if sprels is not None else visn_mask
    v = bert_attention(sd, p + ".visn_self_att", v, m, cfg)
    return ffn(sd, p + ".visn_inter", p + ".visn_output", v, cfg)


def xlayer_lang2visn(sd, p, lang, lang_mask, visn, visn_mask, cfg):  # forward_lang2visn, :400-411
    l = cross_attention(sd, p + ".visual_attention", lang, visn, visn_mask, cfg)
    l = bert_attention(sd, p + ".lang_self_att", l, lang_mask, cfg)
    return ffn(sd, p + ".lang_inter", p + ".lang_output", l, cfg)


def xlayer_visn2visn(sd, p, visn, visn_mask, cfg):  # forward_visn2visn, :413-421
    v = bert_attention(sd, p + ".visn_self_att", visn, visn_mask, cfg)
    return ffn(sd, p + ".visn_inter", p + ".visn_output", v, cfg)


def text_embeddings(sd, txt_ids, cfg):  # BertEmbeddings, :62-77
    p = "bert.embeddings"
    L = txt_ids.shape[1]
    e = sd[p + ".word_embeddings.weight"][txt_ids] + sd[p + ".position_embeddings.weight"][:L][None] + \
        sd[p + ".token_type_embeddings.weight"][0][None, None]
    return _drop(_ln(sd, p + ".LayerNorm", e, cfg.layer_norm_eps), cfg.drop_p)


def language_encoder(sd, txt_embeds, txt_masks, cfg):  # :424-444
    m = neg_mask(txt_masks)
    for i in range(cfg.num_l_layers):
        txt_embeds = bert_layer(sd, "bert.lang_encoder.layer.%d" % i, txt_embeds, m, cfg)
    return txt_embeds if cfg.update_lang_bert else txt_embeds.detach()


def crossmodal_encoder(sd, p, txt, txt_masks, img, img_masks, sprels, cfg):  # :446-463
    tm, im = neg_mask(txt_masks), neg_mask(img_masks)
    for i in range(cfg.num_x_layers):
        img = xlayer_visn(sd, "%s.x_layers.%d" % (p, i), txt, tm, img, im, sprels, cfg)
    return img


# ----------------------------------------------------------------------------- panorama encoder
def pano_layer(sd, p, x, key_pad, cfg):
    """transformer.py:170-182 (pre-norm) with nn.MultiheadAttention's packed in_proj; x is (N, V, H)."""
    H = x.shape[-1]
    h = F.layer_norm(x, (H,), sd[p + ".norm1.weight"], sd[p + ".norm1.bias"], 1e-5)
    qkv = F.linear(h, sd[p + ".self_attn.in_proj_weight"], sd[p + ".self_attn.in_proj_bias"])
    q, k, v = qkv.split(H, dim=-1)
    mask = torch.zeros(key_pad.shape, dtype=torch.float32, device=x.device).masked_fill(key_pad, float("-inf"))
    a = attention_core(q, k, v, mask[:, None, None, :], cfg.num_attention_heads, cfg.drop_p)
    x = x + _drop(_lin(sd, p + ".self_attn.out_proj", a), cfg.drop_p)
    h = F.layer_norm(x, (H,), sd[p + ".norm2.weight"], sd[p + ".norm2.bias"], 1e-5)
    h = _lin(sd, p + ".linear2", _drop(F.gelu(_lin(sd, p + ".linear1", h)), cfg.drop_p))
    return x + _drop(h, cfg.drop_p)


def image_embeddings(sd, b, cfg):  # ImageEmbeddings.forward, vilmodel.py:494-536
    p = "bert.img_embeddings"
    view = _ln(sd, p + ".img_layer_norm", _lin(sd, p + ".img_linear", b["traj_view_img_fts"]), 1e-12)
    if b.get("traj_obj_img_fts") is not None:
        if (p + ".obj_linear.weight") in sd:
            obj = _ln(sd, p + ".obj_layer_norm", _lin(sd, p + ".obj_linear", b["traj_obj_img_fts"]), 1e-12)
        else:
            obj = _ln(sd, p + ".img_layer_norm", _lin(sd, p + ".img_linear", b["traj_obj_img_fts"]), 1e-12)
        vl, ol = b["traj_vp_view_lens"], b["traj_vp_obj_lens"]
        lens = vl + ol
        maxl = int(lens.max())
        rows = []
        for i in range(view.shape[0]):
            r = torch.cat([view[i, : int(vl[i])], obj[i, : int(ol[i])]], 0)
            rows.append(F.pad(r, (0, 0, 0, maxl - r.shape[0])))
        img = torch.stack(rows, 0)
    else:
        img, lens = view, b["traj_vp_view_lens"]
    emb = img + _ln(sd, p + ".loc_layer_norm", _lin(sd, p + ".loc_linear", b["traj_loc_fts"]), 1e-12) + \
        sd[p + ".nav_type_embedding.weight"][b["traj_nav_types"]] + \
        sd["bert.embeddings.token_type_embeddings.weight"][1][None, None]
    emb = _drop(_ln(sd, p + ".layer_norm", emb, 1e-12), cfg.drop_p)
    masks = seq_mask(lens)
    if cfg.num_pano_layers > 0:
        for i in range(cfg.num_pano_layers):
            emb = pano_layer(sd, "%s.pano_encoder.layers.%d" % (p, i), emb, ~masks, cfg)
        emb = _ln(sd, p + ".pano_encoder.norm", emb, 1e-12)
    steps = list(b["traj_step_lens"])
    return torch.split(emb, steps, 0), torch.split(lens, steps, 0)


# ----------------------------------------------------------------------------- global map
def aggregate_gmap(split_embeds, split_lens, b):  # _aggregate_gmap_features, vilmodel.py:632-666
    out = []
    for i, (emb, lens) in enumerate(zip(split_embeds, split_lens)):
        m = seq_mask(lens)
        emb = emb[:, : m.shape[1]] * m[:, :, None]
        visited, unvisited = {}, defaultdict(list)
        for t in range(emb.shape[0]):
            visited[b["traj_vpids"][i][t]] = emb[t].sum(0) / lens[t]
            for j, vp in enumerate(b["traj_cand_vpids"][i][t]):
                if vp not in visited:
                    unvisited[vp].append(emb[t, j])
        rows = []
        for vp in b["gmap_vpids"][i][1:]:
            rows.append(visited[vp] if vp in visited else torch.stack(unvisited[vp], 0).mean(0))
        out.append(torch.stack(rows, 0))
    G = max(r.shape[0] for r in out)
    out = torch.stack([F.pad(r, (0, 0, 0, G - r.shape[0])) for r in out], 0)
    return F.pad(out, (0, 0, 1, 0))  # zero [stop] token first


def gmap_input(sd, split_embeds, split_lens, b):  # gmap_input_embedding, :668-679
    p = "bert.global_encoder"
    g = aggregate_gmap(split_embeds, split_lens, b) + sd[p + ".gmap_step_embeddings.weight"][b["gmap_step_ids"]] + \
        _ln(sd, p + ".gmap_pos_embeddings.1", _lin(sd, p + ".gmap_pos_embeddings.0", b["gmap_pos_fts"]), 1e-12)
    return g, seq_mask(b["gmap_lens"])


def graph_sprels(sd, b):  # vilmodel.py:691-694
    p = "bert.global_encoder.sprel_linear"
    if (p + ".weight") not in sd:
        return None
    d = b["gmap_pair_dists"]
    return (d[..., None] * sd[p + ".weight"].view(1, 1, 1, 1) + sd[p + ".bias"].view(1, 1, 1, 1)).squeeze(3)[:, None]


def bev_input(sd, b):  # LocalBEVEncoder.bev_input_embedding, :589-593
    p = "bert.local_encoder"
    return _ln(sd, p + ".bev_fts_embeddings.1", _lin(sd, p + ".bev_fts_embeddings.0", b["bev_fts"]), 1e-12) + \
        _ln(sd, p + ".bev_pos_embeddings.1", _lin(sd, p + ".bev_pos_embeddings.0", b["bev_pos_fts"]), 1e-12) + \
        sd[p + ".nav_type_embedding.weight"][b["bev_nav_masks"].long()]


def last_obj_tokens(split_embeds, b):  # vilmodel.py:748-756
    if b.get("traj_obj_img_fts") is None:
        return None, None
    steps = list(b["traj_step_lens"])
    vls = [x[-1] for x in torch.split(b["traj_vp_view_lens"], steps, 0)]
    ols = [x[-1] for x in torch.split(b["traj_vp_obj_lens"], steps, 0)]
    rows = [e[-1, int(v): int(v) + int(o)] for e, v, o in zip(split_embeds, vls, ols)]
    mo = max(max(r.shape[0] for r in rows), 0)
    obj = torch.stack([F.pad(r, (0, 0, 0, mo - r.shape[0])) for r in rows], 0)
    return obj, seq_mask(torch.stack(ols, 0), mo) if mo > 0 else torch.zeros(len(rows), 0, dtype=torch.bool)


# ----------------------------------------------------------------------------- BEV lifting
def bevpos_polar(D):  # bev_utils.py:39-58
    lin = torch.linspace(0.5, D - 0.5, D, dtype=torch.float32)
    ry, rx = torch.meshgrid(lin, lin, indexing="ij")
    ry = -(ry - D / 2)
    rx = rx - D / 2
    dis = (ry ** 2 + rx ** 2) ** 0.5
    c, s = rx / dis, ry / dis
    c[dis == 0] = 0
    s[dis == 0] = 0
    return torch.stack([c, s, dis / (D / 2)], -1)


def lift_points(depths, T_c2w, S_w2c, T_w2c, depth_scale=10.0, fx=7.0, fy=7.0, cx=7.0, cy=7.0):
    """pretrain_cmt.py:125-137 + bev_utils.py:130-131,167-171,198: ego-frame point cloud (B,P,3) and the
    no-depth mask (B,P).  The 4-term dot products are evaluated left to right with one rounding per
    operation -- the order the CUDA kernel uses; the reference leaves it to bmm/matmul."""
    B, V = depths.shape[0], depths.shape[1]
    Hf, Wf = depths.shape[-2], depths.shape[-1]
    z = (depths.reshape(B, V, Hf, Wf).to(torch.float32) * depth_scale)
    col = torch.arange(Wf, dtype=torch.float32)
    row = torch.arange(Hf, dtype=torch.float32)
    xs = ((col + 0.5) - cx) / fx
    ys = ((row + 0.5) - cy) / fy
    x = z * xs[None, None, None, :]
    y = z * ys[None, None, :, None]
    T = T_c2w.reshape(B, V, 4, 4)[:, :, :, :, None, None]
    w = []
    for j in range(3):
        acc = T[:, :, j, 0] * x
        acc = acc + T[:, :, j, 1] * y
        acc = acc + T[:, :, j, 2] * z
        acc = acc + T[:, :, j, 3]
        w.append(acc.reshape(B, -1))
    S = S_w2c.reshape(B, 3)
    p = [w[j] - S[:, j: j + 1] for j in range(3)]
    E = T_w2c.reshape(B, 4, 4)
    e = []
    for j in range(3):
        acc = p[0] * E[:, j, 0:1]
        acc = acc + p[1] * E[:, j, 1:2]
        acc = acc + p[2] * E[:, j, 2:3]
        acc = acc + E[:, j, 3:4]
        e.append(acc)
    return torch.stack(e, -1), (z == 0).reshape(B, -1)


def cell_index(pc, no_depth, D, res, y_clip=0.5):
    """bev_utils.py:393-406: (B,P) int64 flat cell index, -1 where the point is dropped."""
    g = (pc[..., [0, 2]] / res + (D - 1) / 2).round()
    outside = (g[..., 0] >= D) | (g[..., 1] >= D) | (g[..., 0] < 0) | (g[..., 1] < 0)
    bad = no_depth | outside | (pc[..., 1] > y_clip)
    idx = (D * g[..., 1] + g[..., 0]).long()
    return torch.where(bad, torch.full_like(idx, -1), idx)


def scatter_mean(src, idx, ncell):
    """torch_scatter.scatter_mean restated (sum in point order, count clamped to 1, true divide)."""
    keep = idx >= 0
    out = torch.zeros((ncell,) + tuple(src.shape[1:]), dtype=src.dtype)
    out.index_add_(0, idx[keep], src[keep])
    cnt = torch.zeros(ncell, dtype=src.dtype)
    cnt.index_add_(0, idx[keep], torch.ones(int(keep.sum()), dtype=src.dtype))
    return out / cnt.clamp(min=1)[:, None]


def lift_splat(b, D, res):
    """pretrain_cmt.py:114-167: consumes the raw grid inputs of `b`, adds bev_* entries (in place)."""
    rgbs, depths, sems = b.pop("rgbs"), b.pop("depths"), b.pop("sems")
    T_c2w, T_w2c, S_w2c, gpos = b.pop("T_c2w"), b.pop("T_w2c"), b.pop("S_w2c"), b.pop("bev_gpos_fts")
    B = rgbs.shape[0]
    pc, nod = lift_points(depths, T_c2w, S_w2c, T_w2c)
    idx = cell_index(pc, nod, D, res)
    feat = rgbs.reshape(B, -1, rgbs.shape[-1])
    sem = sems.reshape(B, -1, sems.shape[-1])
    bev = torch.stack([scatter_mean(feat[i], idx[i], D * D) for i in range(B)], 0)
    bsem = torch.stack([scatter_mean(sem[i], idx[i], D * D) for i in range(B)], 0)
    bsem[bsem > 0] = 1
    b["bev_cell_idx"] = idx
    b["bev_ob_masks"] = ~((bev.max(-1)[0] == 0) & (bev.min(-1)[0] == 0))
    b["bev_fts"] = bev
    b["bev_masks"] = torch.ones(B, D * D, dtype=torch.bool)                     # pretrain_cmt.py:152
    b["bev_pos_fts"] = torch.cat([gpos.expand(-1, D * D, -1), bevpos_polar(D).reshape(1, D * D, 3).expand(B, -1, -1)], -1)
    b["bev_sems"] = bsem
    b["bev_sem_masks"] = bsem.sum(2) > 0
    return b


# ----------------------------------------------------------------------------- model forwards
def _front(sd, b, cfg):
    txt_masks = seq_mask(b["txt_lens"])
    txt = language_encoder(sd, text_embeddings(sd, b["txt_ids"], cfg), txt_masks, cfg)
    split_embeds, split_lens = image_embeddings(sd, b, cfg)
    return txt, txt_masks, split_embeds, split_lens


def _local(sd, b, txt, txt_masks, obj, obj_masks, cfg):  # LocalBEVEncoder.forward, :595-615
    bev = bev_input(sd, b)
    masks = b["bev_masks"]
    if obj is not None:
        bev, masks = torch.cat([bev, obj], 1), torch.cat([masks, obj_masks], 1)
    out = crossmodal_encoder(sd, "bert.local_encoder.encoder", txt, txt_masks, bev, masks, None, cfg)
    n = cfg.bev_dim * cfg.bev_dim
    return out[:, :n], (out[:, n:] if obj is not None else None)


def encode(sd, b, cfg, return_gmap=True):  # GlocalTextPathCMT.forward, :717-765
    txt, txt_masks, se, sl = _front(sd, b, cfg)
    gmap = None
    if return_gmap:
        g, gm = gmap_input(sd, se, sl, b)
        gmap = crossmodal_encoder(sd, "bert.global_encoder.encoder", txt, txt_masks, g, gm, graph_sprels(sd, b), cfg)
    obj, om = last_obj_tokens(se, b)
    bev, obj = _local(sd, b, txt, txt_masks, obj, om, cfg)
    return gmap, bev, obj, om


def encode_mlm(sd, b, cfg):  # GlocalTextPathCMT.forward_mlm, :768-830
    txt, txt_masks, se, sl = _front(sd, b, cfg)
    tm = neg_mask(txt_masks)
    g, gm = gmap_input(sd, se, sl, b)
    gmn = neg_mask(gm)
    gt = txt
    for i in range(cfg.num_x_layers):
        gt = xlayer_lang2visn(sd, "bert.global_encoder.encoder.x_layers.%d" % i, gt, tm, g, gmn, cfg)
    obj, om = last_obj_tokens(se, b)
    bev, masks = bev_input(sd, b), b["bev_masks"]
    if obj is not None:
        bev, masks = torch.cat([bev, obj], 1), torch.cat([masks, om], 1)
    bm = neg_mask(masks)
    bt = txt
    for i in range(cfg.num_x_layers):
        bt = xlayer_lang2visn(sd, "bert.local_encoder.encoder.x_layers.%d" % i, bt, tm, bev, bm, cfg)
    return gt + bt


def encode_sem(sd, b, cfg, mode):  # GlocalTextPathCMT.forward_sem, :833-883
    if mode == "cattn":
        txt, txt_masks, se, sl = _front(sd, b, cfg)
        obj, om = last_obj_tokens(se, b)
        return _local(sd, b, txt, txt_masks, obj, om, cfg)[0]
    bev = bev_input(sd, b)
    if mode == "sattn":
        m = neg_mask(b["bev_masks"])
        for i in range(cfg.num_x_layers):
            bev = xlayer_visn2visn(sd, "bert.local_encoder.encoder.x_layers.%d" % i, bev, m, cfg)
    elif mode != "embed":
        raise NotImplementedError(mode)
    return bev


def _head(sd, p, x):  # Linear -> ReLU -> LN -> Linear, pretrain_cmt.py:34-71
    return _lin(sd, p + ".net.3", _ln(sd, p + ".net.2", F.relu(_lin(sd, p + ".net.0", x)), 1e-12))


def mlm_head(sd, x, cfg):  # vilmodel.py:258-299
    p = "mlm_head.predictions"
    h = _ln(sd, p + ".transform.LayerNorm", _gelu(_lin(sd, p + ".transform.dense", x)), cfg.layer_norm_eps)
    return F.linear(h, sd["bert.embeddings.word_embeddings.weight"]) + sd[p + ".bias"]


def sap_logits(sd, b, cfg, gmap, bev):  # forward_sap, pretrain_cmt.py:322-356
    B = gmap.shape[0]
    if ("sap_fuse_linear.net.0.weight") in sd:
        centre = (cfg.bev_dim * cfg.bev_dim - 1) // 2
        fuse = torch.sigmoid(_head(sd, "sap_fuse_linear", torch.cat([gmap[:, 0], bev[:, centre]], 1)))
    else:
        fuse = 0.5
    gl = _head(sd, "global_sap_head", gmap).squeeze(2) * fuse
    gl = gl.masked_fill(b["gmap_visited_masks"], float("-inf"))
    gl = gl.masked_fill(~seq_mask(b["gmap_lens"]), float("-inf"))
    ar = torch.arange(B)[:, None]
    cand = bev[ar, b["bev_cand_idxs"]]
    cmask = b["bev_nav_masks"][ar, b["bev_cand_idxs"]]
    ll = _head(sd, "local_sap_head", cand).squeeze(2) * (1 - fuse)
    ll = ll.masked_fill(~cmask, float("-inf"))
    rows = [gl[:, 0] + ll[:, 0]]
    fused_cols = {}
    fl = gl.clone()
    fl[:, 0] = rows[0]
    for i in range(B):
        visited = {vp for vp, m in zip(b["gmap_vpids"][i], b["gmap_visited_masks"][i]) if m}
        tmp, bw = {}, 0
        for j, vp in enumerate(b["traj_cand_vpids"][i][-1]):
            if vp in visited:
                bw = bw + ll[i, j + 1]
            else:
                tmp[vp] = ll[i, j + 1]
        for j, vp in enumerate(b["gmap_vpids"][i]):
            if j > 0 and vp not in visited:
                fl[i, j] = fl[i, j] + (tmp[vp] if vp in tmp else bw)
    return gl, ll, fl


def forward(sd, batch, task, cfg, compute_loss=True):
    """GlocalTextPathCMTPreTraining.forward, pretrain_cmt.py:169-238 (+ per-task methods :240-441)."""
    b = dict(batch)
    b = lift_splat(b, cfg.bev_dim, cfg.bev_res)
    if cfg.feat_drop_p > 0:  # drop_feats, :102-106
        for k in ("traj_view_img_fts", "traj_obj_img_fts", "bev_fts"):
            if b.get(k) is not None:
                b[k] = _drop(b[k], cfg.feat_drop_p)
    if task.startswith("mlm"):
        txt = encode_mlm(sd, b, cfg)
        sel = b["txt_labels"] != -1
        scores = mlm_head(sd, txt[sel], cfg)
        return F.cross_entropy(scores, b["txt_labels"][sel], reduction="none") if compute_loss else scores
    if task.startswith("mrc"):
        _, _, obj, _ = encode(sd, b, cfg, return_gmap=False)
        sel = b["vp_obj_mrc_masks"]
        logits, tgt = _head(sd, "obj_classifier", obj[sel]), b["vp_obj_probs"][sel]
        if not compute_loss:
            return logits, tgt
        return F.kl_div(F.log_softmax(logits, -1), tgt, reduction="none").sum(1)
    if task.startswith("sap"):
        gmap, bev, _, _ = encode(sd, b, cfg)
        gl, ll, fl = sap_logits(sd, b, cfg, gmap, bev)
        if not compute_loss:
            return gl, ll, fl, b["global_act_labels"], b["local_act_labels"]
        return F.cross_entropy(gl, b["global_act_labels"], reduction="none") + \
            F.cross_entropy(ll, b["local_act_labels"], reduction="none") + \
            F.cross_entropy(fl, b["global_act_labels"], reduction="none")
    if task.startswith("og"):
        _, _, obj, om = encode(sd, b, cfg, return_gmap=False)
        logits = _head(sd, "og_head", obj).squeeze(2).masked_fill(~om, float("-inf"))
        return F.cross_entropy(logits, b["obj_labels"], reduction="none") if compute_loss else logits
    if task.startswith("sem") or task.startswith("masksem"):
        sel = b["bev_sem_masks"]
        if task.startswith("masksem"):  # :423-424,433
            b["bev_fts"] = b["bev_fts"].masked_fill(b["bev_mrc_masks"][:, :, None], 0)
            sel = sel & b["bev_mrc_masks"]
        bev = encode_sem(sd, b, cfg, cfg.sem_pred_token)
        logits, labels = _head(sd, "local_sem_head", bev[sel]), b["bev_sems"][sel].float()
        if not compute_loss:
            return logits, labels
        return F.binary_cross_entropy_with_logits(logits, labels, reduction="none")
    raise ValueError("invalid task")


class OracleConfig:
    """Attribute bag: the model config keys the path reads (SURVEY.md 5) + oracle knobs."""

    def __init__(self, config, drop_p=0.0, feat_drop_p=0.0, bev_res=None):
        for k in ("hidden_size", "num_attention_heads", "layer_norm_eps", "num_l_layers", "num_x_layers",
                  "num_pano_layers", "bev_dim", "update_lang_bert"):
            setattr(self, k, getattr(config, k))
        self.sem_pred_token = getattr(config, "sem_pred_token", "cattn")
        self.bev_res = bev_res if bev_res is not None else getattr(config, "bev_res", 0.5)
        self.drop_p = drop_p
        self.feat_drop_p = feat_drop_p


# ----------------------------------------------------------------------------- navigation-side API (agents)
def _nav_sd(sd):
    """GlocalTextPathNavCMT keeps the encoder at the top level (no `bert.` prefix); map to the names above."""
    heads = ("global_sap_head", "local_sap_head", "sap_fuse_linear", "og_head")
    return {(k if k.startswith(heads) else "bert." + k): v for k, v in sd.items()}


def nav_forward(sd, mode, batch, cfg):
    """GlocalTextPathNavCMT.forward(mode, batch), map_nav_src/models/vilmodel.py:744-912."""
    sd = _nav_sd(sd)
    if mode == "language":  # forward_text :744-748
        return language_encoder(sd, text_embeddings(sd, batch["txt_ids"], cfg), batch["txt_masks"], cfg)
    if mode == "panorama":  # forward_panorama_per_step :750-801
        b = {"traj_view_img_fts": batch["view_img_fts"], "traj_obj_img_fts": batch.get("obj_img_fts"),
             "traj_loc_fts": batch["loc_fts"], "traj_nav_types": batch["nav_types"],
             "traj_vp_view_lens": batch["view_lens"], "traj_vp_obj_lens": batch.get("obj_lens"),
             "traj_step_lens": [batch["view_img_fts"].shape[0]]}
        (emb,), (lens,) = image_embeddings(sd, b, cfg)
        return emb, seq_mask(lens, emb.shape[1])
    if mode != "navigation":
        raise NotImplementedError(mode)
    # forward_navigation_per_step :803-887
    b = batch
    p = "bert.global_encoder"
    g = b["gmap_img_embeds"] + sd[p + ".gmap_step_embeddings.weight"][b["gmap_step_ids"]] + \
        _ln(sd, p + ".gmap_pos_embeddings.1", _lin(sd, p + ".gmap_pos_embeddings.0", b["gmap_pos_fts"]), 1e-12)
    gmap = crossmodal_encoder(sd, p + ".encoder", b["txt_embeds"], b["txt_masks"], g, b["gmap_masks"],
                              graph_sprels(sd, b), cfg)
    bev, obj = _local(sd, b, b["txt_embeds"], b["txt_masks"], b.get("obj_embeds"), b.get("obj_masks"), cfg)
    sb = {"gmap_visited_masks": b["gmap_visited_masks"], "gmap_lens": b["gmap_masks"].sum(1), "bev_cand_idxs": b["bev_cand_idxs"],
          "bev_nav_masks": b["bev_nav_masks"], "gmap_vpids": b["gmap_vpids"],
          "traj_cand_vpids": [[c[1:]] for c in b["bev_cand_vpids"]]}
    gl, ll, fl = sap_logits(sd, sb, cfg, gmap, bev)
    ol = None
    if obj is not None:
        ol = _head(sd, "og_head", obj).squeeze(2).masked_fill(~b["obj_masks"], float("-inf"))
    return {"gmap_embeds": gmap, "global_logits": gl, "local_logits": ll, "fused_logits": fl, "obj_logits": ol}
