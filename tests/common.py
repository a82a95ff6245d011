"""Shared helpers for the parity tests (TEST code: may import oracle/)."""
import glob
import os

import torch

from etpnav_b200.config import PlannerConfig
from etpnav_b200.synth import make_inputs, make_weights

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
GOLDEN_GRADS_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "grads")

# bf16-operand mode (GEMM / attention operands rounded to bf16, fp32 everywhere else) against the fp32 reference:
# <= 2x the envelope measured on B200 (profiles/r01_parity_report_final.jsonl: logits 0.0037-0.0089, embeddings
# 0.011-0.015).  The strict north_star band (rtol 1e-3 / atol 1e-4) is asserted for precision="high" in
# tests/test_precision_gpu.py.
BF16_LOGIT_TOL = 1.5e-2
BF16_EMBED_TOL = 3e-2
# node selection is asserted bit-exact; the assertion is only meaningful when the fixture's top-2 logit gap is well
# above the measured logit error: fail if gap < NEAR_TIE_FACTOR * max |logit error|
NEAR_TIE_FACTOR = 4.0


def no_dropout(cfg):
    """Parity with the fp32 oracle is defined with dropout off (SURVEY.md §7): zero the three probabilities so that
    train() mode computes the p = 0 function.  tests/test_dropout_gpu.py covers the p > 0 path."""
    cfg.hidden_dropout_prob = cfg.attention_probs_dropout_prob = cfg.pred_head_dropout_prob = 0.0
    return cfg


def golden_names():
    return sorted(os.path.splitext(os.path.basename(p))[0] for p in glob.glob(os.path.join(GOLDEN_DIR, "*.pt")))


def load_case(name):
    """Returns (golden dict, cfg, weights, inputs) with weights/inputs rebuilt from the seeds."""
    gold = torch.load(os.path.join(GOLDEN_DIR, name + ".pt"), weights_only=False)
    c = gold["case"]
    cfg = PlannerConfig(**c["cfg"])
    sd = make_weights(cfg, seed=c["wseed"])
    inp = make_inputs(cfg, c["B"], c["V"], c["N"], c["L"], seed=c["iseed"], ragged=c["ragged"])
    return gold, cfg, sd, inp


def slim(gold, t, key=None):
    """The rows of ``t`` the fixture stores under ``key`` (oracle/make_golden.py: the case's ``slim`` and ``stride``)."""
    c = gold["case"]
    s = (c.get("slim") or 1) * c.get("stride", {}).get(key, 1)
    return t[:, ::s] if (s > 1 and t.dim() == 3) else t


def grad_sig(t):
    t = t.detach().double().flatten()
    return torch.cat([t.sum()[None], t.norm()[None], t[:8]]).float()


def golden_loss(gold, pano, pmask, gmap_embeds, logits, inp):
    """The scalar the fixtures differentiate (oracle/make_golden.py:run_case)."""
    g = torch.Generator().manual_seed(77)
    pw = (torch.randn(pano.shape, generator=g) * pmask.cpu()[..., None]).to(pano)
    gw = (torch.randn(gmap_embeds.shape, generator=g) * inp["gmap_masks"][..., None]).to(gmap_embeds)
    return (torch.nn.functional.cross_entropy(logits, inp["labels"].to(logits.device), reduction="sum")
            + (pano * pw).sum() * 0.01 + (gmap_embeds * gw).sum() * 0.01)
