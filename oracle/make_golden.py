"""Generate tests/golden/*.pt by running the UNMODIFIED reference (authoring container only).

TEST INFRASTRUCTURE.  Usage:  python -m oracle.make_golden
Each fixture stores the case definition (config, shapes, seeds), the reference's fp32 outputs
for forward_txt / forward_panorama / forward_navigation on the seeded synthetic inputs of
``etpnav_b200.synth`` (eval mode, dropout off), the caller-side CE loss, full gradients w.r.t.
the activations that the trainer keeps live (txt_embeds, gmap_img_fts, rgb_fts, dep_fts) and a
compact signature (sum, L2 norm, first 8 values) of the gradient of every parameter.
"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from etpnav_b200.config import PlannerConfig          # noqa: E402
from etpnav_b200.synth import make_inputs, make_weights  # noqa: E402
from oracle import ref_import                          # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

# ``slim``: every slim-th row of all the [B, S, 768] tensors is stored (the tests then feed the nav step their own
# txt_embeds).  ``stride``: of the listed tensors only every stride-th of those rows is stored; txt_embeds is never
# listed, it is the nav step's input in the tests.  Both keep a fixture file under 1 MB.
CASES = {
    # BASELINE.json configs[0]: B=2, 12 views, 16-node graph, 80-token instruction
    "c1_bert": dict(cfg=dict(vocab_size=30522), B=2, V=12, N=16, L=80, ragged=False, wseed=0, iseed=0,
                    stride=dict(grad_txt_embeds=4, grad_gmap_img_fts=2)),
    # ragged lengths everywhere (SURVEY.md Appendix A check shape)
    "ragged_bert": dict(cfg=dict(vocab_size=2048), B=3, V=14, N=11, L=17, ragged=True, wseed=1, iseed=1),
    # XLM-R style eps, no sprels, no depth embedding
    "ragged_xlmr_nosprel_nodepth": dict(
        cfg=dict(vocab_size=2048, max_position_embeddings=514, layer_norm_eps=1e-5,
                 graph_sprels=False, use_depth_embedding=False),
        B=4, V=16, N=24, L=40, ragged=True, wseed=2, iseed=2,
        stride=dict(pano_embeds=2, gmap_embeds=2, grad_txt_embeds=8, grad_rgb_fts=4, grad_gmap_img_fts=4)),
    # a mid-size ragged case with nodes > 64 and text > 128 (two K/V tiles in the attention kernels)
    "mid_bert": dict(cfg=dict(vocab_size=2048, num_l_layers=2), B=5, V=13, N=70, L=150, ragged=True,
                     wseed=3, iseed=3, slim=7, stride=dict(grad_txt_embeds=2)),
}


def grad_sig(t):
    t = t.detach().double().flatten()
    return torch.cat([t.sum()[None], t.norm()[None], t[:8]]).float()


def run_case(name, c):
    cfg = PlannerConfig(**c["cfg"])
    sd = make_weights(cfg, seed=c["wseed"])
    inp = make_inputs(cfg, c["B"], c["V"], c["N"], c["L"], seed=c["iseed"], ragged=c["ragged"])
    ref = ref_import.build_reference(cfg, sd).eval()
    out = {"case": c, "name": name}
    # forward_txt (vilmodel_cmt.py:684) — the nav step then uses ITS output as txt_embeds
    txt = ref.forward_txt(inp["txt_ids"], inp["txt_masks"])
    out["txt_embeds"] = txt.detach().clone()
    leaves = {}
    for k in ("rgb_fts", "dep_fts", "gmap_img_fts"):
        leaves[k] = inp[k].clone().requires_grad_(True)
    txt_leaf = txt.detach().clone().requires_grad_(True)
    pano, pmask = ref.forward_panorama(leaves["rgb_fts"], leaves["dep_fts"], inp["loc_fts"],
                                       inp["nav_types"], inp["view_lens"])
    nav = ref.forward_navigation(txt_leaf, inp["txt_masks"], None, inp["gmap_step_ids"],
                                 leaves["gmap_img_fts"], inp["gmap_pos_fts"], inp["gmap_masks"],
                                 inp["gmap_visited_masks"], inp["gmap_pair_dists"])
    out["pano_embeds"] = pano.detach().clone()
    out["pano_masks"] = pmask.clone()
    out["gmap_embeds"] = nav["gmap_embeds"].detach().clone()
    out["global_logits"] = nav["global_logits"].detach().clone()
    # loss: CE(sum) on the node logits (ss_trainer_ETP.py:890-892) + a pano term so that the
    # panorama branch receives a gradient (the trainer feeds pano_embeds into the map, :838-869)
    g = torch.Generator().manual_seed(77)
    pw = torch.randn(pano.shape, generator=g) * pmask[..., None]
    gw = torch.randn(nav["gmap_embeds"].shape, generator=g) * inp["gmap_masks"][..., None]
    loss = (torch.nn.functional.cross_entropy(nav["global_logits"], inp["labels"], reduction="sum")
            + (pano * pw).sum() * 0.01 + (nav["gmap_embeds"] * gw).sum() * 0.01)
    out["loss"] = loss.detach().clone()
    loss.backward()
    out["grad_txt_embeds"] = txt_leaf.grad.clone()
    for k, v in leaves.items():
        if v.grad is not None:
            out["grad_" + k] = v.grad.clone()
    out["param_grad_sig"] = {k: grad_sig(p.grad) for k, p in ref.named_parameters() if p.grad is not None}
    out["input_sig"] = {k: grad_sig(v.float()) for k, v in inp.items()
                        if isinstance(v, torch.Tensor) and v.dtype.is_floating_point}
    if c.get("slim"):  # keep the fixture small: every slim-th row of the [B,S,768] tensors
        for k in list(out):
            if isinstance(out[k], torch.Tensor) and out[k].dim() == 3:
                out[k] = out[k][:, ::c["slim"]].clone()
    for k, s in c.get("stride", {}).items():
        out[k] = out[k][:, ::s].clone()
    os.makedirs(OUT, exist_ok=True)
    torch.save(out, os.path.join(OUT, name + ".pt"))
    print(name, "loss", float(loss), "logits[0,:4]", nav["global_logits"][0, :4].tolist())


FP64_CASE = "ragged_bert"
FP64_COLS = 64


def run_fp64(name, c):
    """The reference in fp64 on one case -> tests/golden/fp64/<name>.pt: every row of the three embeddings at a fixed
    sample of FP64_COLS hidden columns, the pano masks and all node logits (tests/test_oracle.py holds the fp64 port to
    them).  The nav step consumes the reference's own fp64 txt_embeds, as in the fp32 fixtures."""
    cfg = PlannerConfig(**c["cfg"])
    sd = make_weights(cfg, seed=c["wseed"])
    inp = make_inputs(cfg, c["B"], c["V"], c["N"], c["L"], seed=c["iseed"], ragged=c["ragged"])
    ref = ref_import.build_reference(cfg, sd).double().eval()
    i64 = {k: (v.double() if isinstance(v, torch.Tensor) and v.dtype.is_floating_point else v) for k, v in inp.items()}
    with torch.no_grad():
        txt = ref.forward_txt(i64["txt_ids"], i64["txt_masks"])
        pano, pmask = ref.forward_panorama(i64["rgb_fts"], i64["dep_fts"], i64["loc_fts"], i64["nav_types"],
                                           i64["view_lens"])
        nav = ref.forward_navigation(txt, i64["txt_masks"], None, i64["gmap_step_ids"], i64["gmap_img_fts"],
                                     i64["gmap_pos_fts"], i64["gmap_masks"], i64["gmap_visited_masks"],
                                     i64["gmap_pair_dists"])
    cols = torch.randperm(txt.shape[-1], generator=torch.Generator().manual_seed(64))[:FP64_COLS].sort().values
    out = {"case": c, "name": name, "cols": cols, "txt_embeds": txt[..., cols].clone(),
           "pano_embeds": pano[..., cols].clone(), "pano_masks": pmask.clone(),
           "gmap_embeds": nav["gmap_embeds"][..., cols].clone(), "global_logits": nav["global_logits"].clone()}
    os.makedirs(os.path.join(OUT, "fp64"), exist_ok=True)
    torch.save(out, os.path.join(OUT, "fp64", name + ".pt"))
    print(name, "fp64 logits[0,:4]", nav["global_logits"][0, :4].tolist())


if __name__ == "__main__":
    assert ref_import.available(), "reference not mounted"
    torch.manual_seed(0)
    for name, c in CASES.items():
        run_case(name, c)
    run_fp64(FP64_CASE, CASES[FP64_CASE])
