"""Generate tests/golden/pretrain/*.pt by running the UNMODIFIED reference pre-training model (oracle/ref_import.py).

TEST INFRASTRUCTURE.  Usage:  python -m oracle.make_golden_pretrain
Each fixture stores the case definition (config, shapes, seeds) and what ``GlocalTextPathCMTPreTraining``
(pretrain_src/pretrain_src/model/pretrain_cmt.py:50) returns in eval mode on the seeded synthetic batch of
``etpnav_b200.synth.make_traj_batch``: the twin's ``forward`` (gmap_embeds) and ``forward_mlm`` (txt_embeds), the ``sap``
logits / losses, the ``mlm`` scores / losses, and — for loss = mean(mlm) + mean(sap) — the gradient w.r.t. the view
features plus a signature (sum, L2 norm, first 8 values) of every parameter gradient.
"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from etpnav_b200.config import PlannerConfig              # noqa: E402
from etpnav_b200.synth import make_traj_batch, make_weights  # noqa: E402
from oracle import ref_import                              # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "pretrain")
_PT = dict(use_lang2visn_attn=True, mlm_head=True)

CASES = {
    "pt_small": dict(cfg=dict(vocab_size=2048, num_l_layers=2, num_x_layers=2, **_PT), B=3, T=3, V=8, L=20, ghosts=3,
                     wseed=5, iseed=5),
    # more views than the navigation model ever sees (36 = the pre-training panorama), text longer than one 128-row
    # query tile, a map with two dozen nodes, XLM-R style eps and no sprels
    "pt_mid": dict(cfg=dict(vocab_size=2048, num_l_layers=2, num_x_layers=3, max_position_embeddings=514,
                            layer_norm_eps=1e-5, graph_sprels=False, **_PT), B=4, T=6, V=36, L=150, ghosts=16,
                   wseed=6, iseed=6, slim=6),
}


def grad_sig(t):
    t = t.detach().double().flatten()
    return torch.cat([t.sum()[None], t.norm()[None], t[:8]]).float()


def twin_args(b):
    return (b["txt_ids"], b["txt_lens"], b["traj_view_img_fts"], b["traj_view_dep_fts"], b["traj_obj_img_fts"],
            b["traj_loc_fts"], b["traj_nav_types"], b["traj_step_lens"], b["traj_vp_view_lens"], b["traj_vp_obj_lens"],
            b["traj_vpids"], b["traj_cand_vpids"], b["gmap_lens"], b["gmap_step_ids"], b["gmap_pos_fts"],
            b["gmap_pair_dists"], b["gmap_vpids"])


def run_case(name, c):
    cfg = PlannerConfig(**c["cfg"])
    sd = make_weights(cfg, seed=c["wseed"])
    b = make_traj_batch(cfg, c["B"], c["T"], c["V"], c["L"], seed=c["iseed"], ghosts=c["ghosts"])
    ref = ref_import.build_pretrain_reference(cfg, sd).eval()
    out = {"case": c, "name": name}
    b = dict(b)
    b["traj_view_img_fts"] = b["traj_view_img_fts"].clone().requires_grad_(True)
    out["gmap_embeds"] = ref.bert(*twin_args(b)).detach().clone()
    out["mlm_txt_embeds"] = ref.bert.forward_mlm(*twin_args(b)).detach().clone()
    logits, _ = ref(b, "sap", compute_loss=False)
    out["sap_logits"] = logits.detach().clone()
    out["mlm_scores"] = ref(b, "mlm", compute_loss=False).detach().clone()
    sap = ref(b, "sap", compute_loss=True)
    mlm = ref(b, "mlm", compute_loss=True)
    out["sap_loss"], out["mlm_loss"] = sap.detach().clone(), mlm.detach().clone()
    (mlm.mean() + sap.mean()).backward()
    out["grad_traj_view_img_fts"] = b["traj_view_img_fts"].grad.clone()
    sig = {}
    for k, p in ref.named_parameters():
        if p.grad is not None:
            sig[k[5:] if k.startswith("bert.") else k] = grad_sig(p.grad)
    out["param_grad_sig"] = sig
    if c.get("slim"):
        for k in ("gmap_embeds", "mlm_txt_embeds", "grad_traj_view_img_fts"):
            out[k] = out[k][:, ::c["slim"]].clone()
        out["mlm_scores"] = out["mlm_scores"][:, ::c["slim"]].clone()
    os.makedirs(OUT, exist_ok=True)
    torch.save(out, os.path.join(OUT, name + ".pt"))
    print(name, "sap", sap.tolist(), "mlm[:3]", mlm[:3].tolist(), "N", b["gmap_step_ids"].shape[1],
          "masked", int((b["txt_labels"] != -1).sum()))


if __name__ == "__main__":
    assert ref_import.available(), "reference not mounted"
    torch.manual_seed(0)
    for name, c in CASES.items():
        run_case(name, c)
