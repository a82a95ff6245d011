"""CPU restatement of the PRE-TRAINING twin of the planner — TEST INFRASTRUCTURE, not product code.

Restates ``GlocalTextPathCMT`` / ``GlocalTextPathCMTPreTraining`` (paths relative to
/root/reference/pretrain_src/pretrain_src/model) in plain tensor algebra on the raw ``state_dict`` (keys in the planner
namespace, i.e. without the ``bert.`` prefix), reusing ``oracle/planner_port.py`` for the layers both models share.
Pinned by ``oracle/make_golden_pretrain.py`` (the UNMODIFIED reference run in the authoring container on seeded
synthetic batches -> ``tests/golden/pretrain/*.pt``) and ``tests/test_oracle_pretrain.py``.
"""
import torch
import torch.nn.functional as F

from . import planner_port as P


def seq_masks(lens, width):
    # ops.py:37-45 (gen_seq_masks); the collate pads to max(lens) so width == max(lens)
    return torch.arange(width, device=lens.device)[None] < lens[:, None]


def img_embeddings(sd, cfg, b, drop=None):
    """ImageEmbeddings.forward (vilmodel.py:488-534) without object features: the same packing + pano encoder as the
    navigation model's forward_panorama, over the [sum(steps), V, *] trajectory batch; returns the per-episode splits."""
    x, _ = P.forward_panorama(sd, cfg, b["traj_view_img_fts"], b["traj_view_dep_fts"], b["traj_loc_fts"],
                              b["traj_nav_types"], b["traj_vp_view_lens"], drop)
    return torch.split(x, b["traj_step_lens"], 0), torch.split(b["traj_vp_view_lens"], b["traj_step_lens"], 0)


def aggregate_gmap_features(split_embeds, split_lens, traj_vpids, traj_cand_vpids, gmap_vpids):
    """GlobalMapEncoder._aggregate_gmap_features (vilmodel.py:585-619), loop for loop."""
    out = []
    for i in range(len(split_embeds)):
        visited, unvisited = {}, {}
        lens = split_lens[i]
        e = split_embeds[i][:, :int(lens.max())] * seq_masks(lens, int(lens.max()))[..., None]
        for t in range(len(split_embeds[i])):
            visited[traj_vpids[i][t]] = e[t].sum(0) / lens[t]
            for j, vp in enumerate(traj_cand_vpids[i][t]):
                if vp not in visited:
                    unvisited.setdefault(vp, []).append(e[t][j])
        rows = [visited[vp] if vp in visited else torch.stack(unvisited[vp], 0).mean(0) for vp in gmap_vpids[i][1:]]
        out.append(torch.stack(rows, 0))
    n = max(len(r) for r in out)
    H = out[0].shape[1]
    pad = torch.zeros(len(out), n + 1, H, dtype=out[0].dtype)   # [stop] token first (:613-617), zero padding
    for i, r in enumerate(out):
        pad[i, 1:1 + len(r)] = r
    return pad


def gmap_input_embedding(sd, gmap_img_fts, gmap_step_ids, gmap_pos_fts):
    # vilmodel.py:621-632
    return (gmap_img_fts + sd["global_encoder.gmap_step_embeddings.weight"][gmap_step_ids]
            + P._ln(sd, "global_encoder.gmap_pos_embeddings.1",
                    P._lin(sd, "global_encoder.gmap_pos_embeddings.0", gmap_pos_fts), 1e-12))


def _txt(sd, cfg, b, drop=None):
    txt_masks = seq_masks(b["txt_lens"], b["txt_ids"].shape[1])
    return P.forward_txt(sd, cfg, b["txt_ids"], txt_masks, drop), txt_masks   # vilmodel.py:673-676


def forward_gmap(sd, cfg, b, drop=None):
    """GlocalTextPathCMT.forward (vilmodel.py:668-711) + the SAP logits of forward_sap (pretrain_cmt.py:229-233)."""
    txt, txt_masks = _txt(sd, cfg, b, drop)
    se, sl = img_embeddings(sd, cfg, b, drop)
    img = aggregate_gmap_features(se, sl, b["traj_vpids"], b["traj_cand_vpids"], b["gmap_vpids"])
    gm = seq_masks(b["gmap_lens"], b["gmap_step_ids"].shape[1])
    vis = b.get("gmap_visited_masks")
    if vis is None:
        vis = torch.zeros_like(gm)
    return P.forward_navigation(sd, cfg, txt, txt_masks, None, b["gmap_step_ids"], img, b["gmap_pos_fts"], gm, vis,
                                b["gmap_pair_dists"], drop)


SITE_L2V = 4000


def forward_mlm(sd, cfg, b, drop=None):
    """GlocalTextPathCMT.forward_mlm (vilmodel.py:713-754): GraphLXRTXLayer.forward_lang2visn (:400-411) per x-layer."""
    txt, txt_masks = _txt(sd, cfg, b, drop)
    se, sl = img_embeddings(sd, cfg, b, drop)
    img = aggregate_gmap_features(se, sl, b["traj_vpids"], b["traj_cand_vpids"], b["gmap_vpids"])
    nodes = gmap_input_embedding(sd, img, b["gmap_step_ids"], b["gmap_pos_fts"])
    gm = seq_masks(b["gmap_lens"], b["gmap_step_ids"].shape[1])
    dt = txt.dtype
    tbias, nbias = P.extend_neg_masks(txt_masks, dt), P.extend_neg_masks(gm, dt)
    h, eps = cfg.num_attention_heads, cfg.layer_norm_eps
    x = txt
    for i in range(cfg.num_x_layers):
        p = f"global_encoder.encoder.x_layers.{i}."
        ctx = P._bert_ctx(sd, p + "visual_attention.att.", x, nodes, nbias, h, drop, P._site(SITE_L2V, i, P.K_XATTN))
        o = P._drop(drop, P._lin(sd, p + "visual_attention.output.dense", ctx), "hidden", P._site(SITE_L2V, i, P.K_XOUT))
        a = P._ln(sd, p + "visual_attention.output.LayerNorm", o + x, eps)
        ctx = P._bert_ctx(sd, p + "lang_self_att.self.", a, a, tbias, h, drop, P._site(SITE_L2V, i, P.K_SATTN))
        o = P._drop(drop, P._lin(sd, p + "lang_self_att.output.dense", ctx), "hidden", P._site(SITE_L2V, i, P.K_SOUT))
        c = P._ln(sd, p + "lang_self_att.output.LayerNorm", o + a, eps)
        f = P._lin(sd, p + "lang_output.dense", P.gelu_erf(P._lin(sd, p + "lang_inter.dense", c)))
        f = P._drop(drop, f, "hidden", P._site(SITE_L2V, i, P.K_FFNOUT))
        x = P._ln(sd, p + "lang_output.LayerNorm", f + c, eps)
    return x


def mlm_head(sd, cfg, hidden):
    """BertOnlyMLMHead (vilmodel.py:258-299), decoder tied to the word embeddings (pretrain_cmt.py:79-82)."""
    t = P.gelu_erf(P._lin(sd, "mlm_head.predictions.transform.dense", hidden))
    t = P._ln(sd, "mlm_head.predictions.transform.LayerNorm", t, cfg.layer_norm_eps)
    return t @ sd["embeddings.word_embeddings.weight"].t() + sd["mlm_head.predictions.bias"]


def task_mlm(sd, cfg, b, compute_loss=True, drop=None):
    """GlocalTextPathCMTPreTraining.forward_mlm (pretrain_cmt.py:137-164)."""
    x = forward_mlm(sd, cfg, b, drop)
    mask = b["txt_labels"] != -1
    scores = mlm_head(sd, cfg, x[mask])
    if compute_loss:
        return F.cross_entropy(scores, b["txt_labels"][mask], reduction="none")
    return scores


def task_sap(sd, cfg, b, compute_loss=True, drop=None):
    """GlocalTextPathCMTPreTraining.forward_sap (pretrain_cmt.py:218-262)."""
    logits = forward_gmap(sd, cfg, b, drop)["global_logits"]
    if compute_loss:
        return F.cross_entropy(logits, b["global_act_labels"], reduction="none")
    return logits, b["global_act_labels"]
