"""Generate tests/golden/grads/c1_bert.pt by running the UNMODIFIED reference (oracle/ref_import.py).

TEST INFRASTRUCTURE.  Usage:  python -m oracle.make_golden_grads
The c1_bert fixture of tests/golden stores a 10-number signature per parameter gradient.  A full copy of the 140 M
gradients would be 563 MB, so this companion fixture stores, for every parameter of the pano / nav groups (the ones the
planner step trains), a SKETCH of the reference's fp32 gradient that pins every region of the tensor:
  1-D tensors: the full gradient;
  2-D tensors: all row sums, all column sums and 64 single entries (flat indices drawn from a fixed generator).
A sign or indexing error confined to a slice of a weight gradient (one head, one k-block, one output tile) moves the
row / column sums of that slice; tests/test_backward_gpu.py compares every vector.  The sketch stays under 1 MB.
"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from etpnav_b200.config import PlannerConfig          # noqa: E402
from etpnav_b200.synth import make_inputs, make_weights  # noqa: E402
from oracle import ref_import                          # noqa: E402
from oracle.make_golden import CASES                   # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "grads")
TEXT_PREFIXES = ("lang_encoder", "embeddings.word", "embeddings.position", "embeddings.LayerNorm")
SAMPLE = 64     # single entries per 2-D gradient


def sketch_entries(shape, name):
    g = torch.Generator().manual_seed(sum(map(ord, name)) + 123)
    return torch.randint(0, shape[0] * shape[1], (SAMPLE,), generator=g)


def sketch(name, grad):
    g = grad.detach().float()
    if g.dim() < 2:
        return {"full": g.clone()}
    g2 = g.reshape(g.shape[0], -1)
    idx = sketch_entries(g2.shape, name)
    return {"row_sum": g2.double().sum(1).float(), "col_sum": g2.double().sum(0).float(), "idx": idx,
            "vals": g2.flatten()[idx].clone()}


def run(name="c1_bert"):
    c = CASES[name]
    cfg = PlannerConfig(**c["cfg"])
    sd = make_weights(cfg, seed=c["wseed"])
    inp = make_inputs(cfg, c["B"], c["V"], c["N"], c["L"], seed=c["iseed"], ragged=c["ragged"])
    ref = ref_import.build_reference(cfg, sd).eval()
    txt = ref.forward_txt(inp["txt_ids"], inp["txt_masks"]).detach()
    pano, pmask = ref.forward_panorama(inp["rgb_fts"], inp["dep_fts"], inp["loc_fts"], inp["nav_types"], inp["view_lens"])
    nav = ref.forward_navigation(txt, inp["txt_masks"], None, inp["gmap_step_ids"], inp["gmap_img_fts"], inp["gmap_pos_fts"],
                                 inp["gmap_masks"], inp["gmap_visited_masks"], inp["gmap_pair_dists"])
    g = torch.Generator().manual_seed(77)   # the loss of oracle/make_golden.py:run_case
    pw = torch.randn(pano.shape, generator=g) * pmask[..., None]
    gw = torch.randn(nav["gmap_embeds"].shape, generator=g) * inp["gmap_masks"][..., None]
    loss = (torch.nn.functional.cross_entropy(nav["global_logits"], inp["labels"], reduction="sum")
            + (pano * pw).sum() * 0.01 + (nav["gmap_embeds"] * gw).sum() * 0.01)
    loss.backward()
    out = {"case": name, "loss": loss.detach().clone(), "sketch": {}}
    for k, p in ref.named_parameters():
        if p.grad is None or k.startswith(TEXT_PREFIXES):
            continue
        out["sketch"][k] = sketch(k, p.grad)
    os.makedirs(OUT, exist_ok=True)
    torch.save(out, os.path.join(OUT, name + ".pt"))
    print(name, "loss", float(loss), "tensors", len(out["sketch"]))


if __name__ == "__main__":
    assert ref_import.available(), "reference not mounted"
    run()
