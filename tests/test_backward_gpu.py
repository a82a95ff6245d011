"""GPU: backward parity of the step-level CUDA path (autograd through B200Planner) against the gradients the
unmodified reference produced for the golden fixtures (fp32 autograd, oracle/make_golden.py), plus the fused
trainer.  bf16 GEMM operands in forward AND backward: gradients are compared in relative L2 norm.

Tolerance calibration (measured in the authoring container): the REFERENCE ITSELF under
``torch.autocast("cpu", dtype=torch.bfloat16)`` against its own fp32 gradients on the same fixtures gives
relative L2 errors of d_txt_embeds 0.9 % (c1_bert) / 6.1 % (ragged_bert) / 3.3 % (ragged_xlmr), d_gmap_img_fts
0.7 % / 5.6 % / 2.9 %, d_rgb_fts 0.4 %; this path measures 0.9 % / 4.5 % / 4.1 % for d_txt_embeds (B200, round 1).
The bounds below sit just above the reference's own bf16 error."""
import json
import os

import pytest
import torch

from tests.common import golden_loss, golden_names, grad_sig, load_case, no_dropout, slim

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(300)]
REL_L2_ACT = 8e-2     # activations' gradients: ||g - g_ref|| / ||g_ref||
REL_NORM_PARAM = 1e-1  # parameter-gradient norm
REPORT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out", "parity_report.jsonl")


def _rel(a, b):
    return ((a - b).norm() / b.norm().clamp_min(1e-12)).item()


@pytest.mark.parametrize("name", golden_names())
def test_backward_matches_golden(name):
    from etpnav_b200.planner import B200Planner
    gold, cfg, sd, inp = load_case(name)
    no_dropout(cfg)
    m = B200Planner(cfg, device="cuda")
    m.load_state_dict(sd, strict=True)
    m.train()
    d = {k: (v.cuda() if isinstance(v, torch.Tensor) else v) for k, v in inp.items()}
    leaves = {k: d[k].clone().requires_grad_(True) for k in ("rgb_fts", "dep_fts", "gmap_img_fts")}
    if gold["case"].get("slim"):
        with torch.no_grad():
            txt0 = m.forward_txt(d["txt_ids"], d["txt_masks"])
    else:
        txt0 = gold["txt_embeds"].cuda()
    txt_leaf = txt0.detach().clone().requires_grad_(True)
    pano, pm = m.forward_panorama(leaves["rgb_fts"], leaves["dep_fts"], d["loc_fts"], d["nav_types"], d["view_lens"])
    nav = m.forward_navigation(txt_leaf, d["txt_masks"], None, d["gmap_step_ids"], leaves["gmap_img_fts"],
                               d["gmap_pos_fts"], d["gmap_masks"], d["gmap_visited_masks"], d["gmap_pair_dists"])
    loss = golden_loss(gold, pano, pm, nav["gmap_embeds"], nav["global_logits"], inp)
    loss.backward()
    torch.cuda.synchronize()
    rep = {"case": name, "kind": "backward", "loss_err": abs(loss.item() - gold["loss"].item())}
    assert abs(loss.item() - gold["loss"].item()) < 2e-2 * max(1.0, abs(gold["loss"].item()))
    if not gold["case"].get("slim"):
        rep["d_txt"] = _rel(slim(gold, txt_leaf.grad.cpu(), "grad_txt_embeds"), gold["grad_txt_embeds"])
        assert rep["d_txt"] < REL_L2_ACT, rep
    for k, v in leaves.items():
        if "grad_" + k in gold:
            rep["d_" + k] = _rel(slim(gold, v.grad.cpu(), "grad_" + k), gold["grad_" + k])
            assert rep["d_" + k] < REL_L2_ACT, rep
    worst = ("", 0.0)
    for k, sig in gold["param_grad_sig"].items():
        if k.startswith(("lang_encoder", "embeddings.word", "embeddings.position", "embeddings.LayerNorm")):
            continue
        g = m._pmap[k].grad
        assert g is not None, k
        got = grad_sig(g.cpu())
        ref_norm = float(sig[1])
        if ref_norm < 1e-6:   # analytically-zero gradients (sprel bias: softmax shift invariance)
            assert float(got[1]) < 1e-2, (k, got)  # bf16 rounding noise only
            continue
        e = abs(float(got[1]) - ref_norm) / ref_norm
        e8 = float((got[2:] - sig[2:]).abs().max()) / max(float(sig[2:].abs().max()), 1e-3 * ref_norm)
        if max(e, 0.2 * e8) > worst[1]:
            worst = (k, max(e, 0.2 * e8))
        assert e < REL_NORM_PARAM, (k, float(got[1]), ref_norm)
        assert e8 < 0.25, (k, got, sig)
    rep["worst_param"] = worst
    os.makedirs(os.path.dirname(REPORT), exist_ok=True)
    with open(REPORT, "a") as f:
        f.write(json.dumps(rep) + "\n")


def test_parameter_gradients_full_tensors_c1():
    """Every parameter gradient of the c1_bert fixture as a FULL tensor: (i) against the fp32 oracle port run here on the
    same inputs (the port's gradients are pinned to the reference's by tests/test_oracle.py), relative L2 and cosine per
    tensor; (ii) against the gradient sketches of the UNMODIFIED reference (tests/golden/grads, oracle/make_golden_grads.py:
    all row sums, all column sums, 64 sampled entries per matrix; full 1-D tensors) — a sign or indexing error confined to any
    slice of a weight gradient moves its row / column sums."""
    from etpnav_b200.planner import B200Planner
    from oracle import planner_port as P
    from oracle.make_golden_grads import TEXT_PREFIXES
    from tests.common import GOLDEN_GRADS_DIR
    gold, cfg, sd, inp = load_case("c1_bert")
    no_dropout(cfg)
    sk = torch.load(os.path.join(GOLDEN_GRADS_DIR, "c1_bert.pt"), weights_only=False)
    m = B200Planner(cfg, device="cuda")
    m.load_state_dict(sd, strict=True)
    m.train()
    d = {k: (v.cuda() if isinstance(v, torch.Tensor) else v) for k, v in inp.items()}
    txt = gold["txt_embeds"].cuda()
    pano, pm = m.forward_panorama(d["rgb_fts"], d["dep_fts"], d["loc_fts"], d["nav_types"], d["view_lens"])
    nav = m.forward_navigation(txt, d["txt_masks"], None, d["gmap_step_ids"], d["gmap_img_fts"], d["gmap_pos_fts"],
                               d["gmap_masks"], d["gmap_visited_masks"], d["gmap_pair_dists"])
    golden_loss(gold, pano, pm, nav["gmap_embeds"], nav["global_logits"], inp).backward()
    sdc = {k: (v.cuda().clone().requires_grad_(True) if not k.startswith(TEXT_PREFIXES) else v.cuda()) for k, v in sd.items()}
    pano_o, pm_o = P.forward_panorama(sdc, cfg, d["rgb_fts"], d["dep_fts"], d["loc_fts"], d["nav_types"], d["view_lens"])
    nav_o = P.forward_navigation(sdc, cfg, txt, d["txt_masks"], None, d["gmap_step_ids"], d["gmap_img_fts"], d["gmap_pos_fts"],
                                 d["gmap_masks"], d["gmap_visited_masks"], d["gmap_pair_dists"])
    golden_loss(gold, pano_o, pm_o, nav_o["gmap_embeds"], nav_o["global_logits"], inp).backward()
    torch.cuda.synchronize()
    checked, worst = 0, ("", 0.0)
    for k, ref in sk["sketch"].items():
        g = m._pmap[k].grad
        assert g is not None, k
        go = sdc[k].grad
        # (i) full tensor vs the oracle
        if go.norm() < 1e-6:
            assert g.norm() < 1e-2, k     # analytically zero (key biases, sprel bias): bf16 noise only
            continue
        r = _rel(g, go)
        cos = torch.nn.functional.cosine_similarity(g.flatten().double(), go.flatten().double(), dim=0).item()
        worst = max(worst, (k, r), key=lambda t: t[1])
        lim = 0.25 if go.numel() == 1 else REL_NORM_PARAM
        assert r < lim and cos > 1 - lim * lim, (k, r, cos)
        # (ii) sketch of the unmodified reference's gradient
        gc = g.detach().float().cpu()
        if "full" in ref:
            assert _rel(gc, ref["full"]) < lim, (k, "full")
        else:
            g2 = gc.reshape(gc.shape[0], -1)
            R = g2.shape[0]
            # bf16 rounding errors are independent per element: summed over a row / column they grow like the sum of
            # independent entries would, so every vector is measured against max(|reference vector|, the norm the vector
            # would have if the summed entries had random signs) — this keeps analytically-cancelling sums (columns of a
            # weight feeding a LayerNorm sum to ~0) from turning rounding noise into a huge relative error
            row_norm = g2.norm().item() / R ** 0.5
            for name, got, want, floor in (("row_sum", g2.double().sum(1).float(), ref["row_sum"], row_norm * R ** 0.5),
                                           ("col_sum", g2.double().sum(0).float(), ref["col_sum"], row_norm * R ** 0.5),
                                           ("entries", g2.flatten()[ref["idx"]], ref["vals"],
                                            row_norm * (ref["idx"].numel() / g2.shape[1]) ** 0.5)):
                err = (got - want).norm().item()
                assert err < 1.5 * lim * max(want.norm().item(), floor, 1e-12), (k, name, err, want.norm().item(), floor)
        checked += 1
    assert checked >= 140, checked
    with open(REPORT, "a") as f:
        f.write(json.dumps({"case": "c1_bert", "kind": "full_param_grads", "tensors": checked, "worst_rel_l2": worst}) + "\n")


def test_txt_backward_matches_oracle():
    """forward_txt backward (language encoder, SURVEY.md §8f N1) against the fp32 oracle port."""
    from etpnav_b200.config import PlannerConfig
    from etpnav_b200.planner import B200Planner
    from etpnav_b200.synth import make_inputs, make_weights
    from oracle import planner_port as P
    cfg = no_dropout(PlannerConfig(vocab_size=2048, num_l_layers=2))
    sd = make_weights(cfg, seed=21)
    inp = make_inputs(cfg, 3, 12, 8, 37, seed=21, ragged=True)
    m = B200Planner(cfg, device="cuda")
    m.load_state_dict(sd, strict=True)
    m.train()
    g = torch.Generator().manual_seed(5)
    w = torch.randn(3, 37, 768, generator=g) * inp["txt_masks"][..., None]
    out = m.forward_txt(inp["txt_ids"].cuda(), inp["txt_masks"].cuda())
    (out * w.cuda()).sum().backward()
    sdr = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    ref = P.forward_txt(sdr, cfg, inp["txt_ids"], inp["txt_masks"])
    (ref * w).sum().backward()
    for k in sdr:
        if not (k.startswith("lang_encoder") or k.startswith("embeddings")):
            continue
        gr, gg = sdr[k].grad, m._pmap[k].grad
        if gr is None or gr.norm() < 1e-5:   # absent, or analytically zero (key bias: softmax shift invariance)
            continue
        assert gg is not None, k
        assert _rel(gg.cpu(), gr) < 6e-2, (k, _rel(gg.cpu(), gr))


def test_trainer_step_reduces_loss_and_matches_adamw():
    from etpnav_b200.config import PlannerConfig
    from etpnav_b200.planner import B200Planner
    from etpnav_b200.synth import make_inputs, make_weights
    cfg = no_dropout(PlannerConfig(vocab_size=2048, num_l_layers=0, num_x_layers=2))
    sd = make_weights(cfg, seed=8)
    inp = make_inputs(cfg, 8, 12, 20, 30, seed=8, ragged=True)
    d = {k: (v.cuda() if isinstance(v, torch.Tensor) else v) for k, v in inp.items()}
    # (a) fused trainer: loss goes down on a fixed batch
    m = B200Planner(cfg, device="cuda")
    m.load_state_dict(sd, strict=True)
    m.train()
    tr = m.make_trainer(lr=2e-4)
    losses = []
    for _ in range(6):
        tr.zero_grad()
        _, loss = tr.forward_backward(d)
        tr.optimizer_step()
        losses.append(loss.item())
    assert losses[-1] < losses[0], losses
    # (b) one fused AdamW step == torch.optim.AdamW on the same gradients
    m1 = B200Planner(cfg, device="cuda"); m1.load_state_dict(sd, strict=True); m1.train()
    m2 = B200Planner(cfg, device="cuda"); m2.load_state_dict(sd, strict=True); m2.train()
    t1 = m1.make_trainer(lr=1e-3)
    t1.zero_grad(); t1.forward_backward(d)
    grads = m1._direct_grad.clone()
    t1.optimizer_step()
    opt = torch.optim.AdamW([p for p in m2.parameters()], lr=1e-3)
    for n, p in m2._pmap.items():
        off, numel, shape = m2.layout.entries[n]
        p.grad = grads[off:off + numel].view(shape).clone()
    opt.step()
    lo, hi = t1.lo, t1.hi
    assert (m1._flat[lo:hi] - m2._flat[lo:hi]).abs().max() < 1e-6
    assert torch.equal(m1._flat_bf16[lo:hi], m1._flat[lo:hi].bfloat16())
