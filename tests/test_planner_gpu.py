"""GPU: step-level parity of B200Planner (CUDA path through the C ABI) against the golden fixtures
minted from the unmodified reference (tests/golden, oracle/make_golden.py) and against the fp32 oracle
restatement on the same seeded inputs.

Tolerances.  BASELINE.json's north_star asks for rtol=1e-3/atol=1e-4 "bf16".  SURVEY.md §7 measured that
the reference's OWN bf16-autocast path only puts 12-15 % of the logits inside that band against its
fp32 path (max|d| 0.013): bf16 GEMM operands (2^-8 round-off) cannot meet it.  These tests therefore
assert (a) bit-exact node selection (argmax) and -inf pattern, (b) the error of the bf16-operand /
fp32-everything-else kernels against the fp32 reference stays below MAX_ABS_* (measured, recorded in
DESIGN.md), and report the fraction of logits inside the north_star band.
"""
import json
import os

import pytest
import torch

from tests.common import BF16_EMBED_TOL, BF16_LOGIT_TOL, NEAR_TIE_FACTOR, golden_names, load_case, slim

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(300)]

MAX_ABS_EMBED = BF16_EMBED_TOL   # residual-stream embeddings have |x| ~ 1..3 after LayerNorm
MAX_ABS_LOGIT = BF16_LOGIT_TOL
REPORT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out", "parity_report.jsonl")


def _model(cfg, sd):
    from etpnav_b200.planner import B200Planner
    m = B200Planner(cfg, device="cuda")
    missing, unexpected = m.load_state_dict(sd, strict=True)
    return m.eval()


def _cuda(inp):
    return {k: (v.cuda() if isinstance(v, torch.Tensor) else v) for k, v in inp.items()}


def _report(**kw):
    os.makedirs(os.path.dirname(REPORT), exist_ok=True)
    with open(REPORT, "a") as f:
        f.write(json.dumps(kw) + "\n")


@pytest.mark.parametrize("name", golden_names())
def test_forward_matches_golden(name):
    gold, cfg, sd, inp = load_case(name)
    m = _model(cfg, sd)
    d = _cuda(inp)
    with torch.no_grad():
        txt = m.forward_txt(d["txt_ids"], d["txt_masks"])
        pano, pmask = m.forward_panorama(d["rgb_fts"], d["dep_fts"], d["loc_fts"], d["nav_types"], d["view_lens"])
        # like the fixture: the nav step consumes the reference's own txt_embeds (isolates the nav path) ...
        txt_ref = gold["txt_embeds"].cuda() if not gold["case"].get("slim") else txt
        nav = m.forward_navigation(txt_ref, d["txt_masks"], None, d["gmap_step_ids"], d["gmap_img_fts"],
                                   d["gmap_pos_fts"], d["gmap_masks"], d["gmap_visited_masks"], d["gmap_pair_dists"])
    torch.cuda.synchronize()
    tm = inp["txt_masks"]
    e_txt = (slim(gold, txt.cpu(), "txt_embeds") - gold["txt_embeds"]).abs()
    e_txt_valid = (e_txt[slim(gold, tm[..., None].expand_as(txt), "txt_embeds")[..., 0]] if not gold["case"].get("slim")
                   else e_txt)
    assert torch.equal(pmask.cpu(), gold["pano_masks"])
    e_pano = (slim(gold, pano.cpu(), "pano_embeds") - gold["pano_embeds"]).abs()
    e_emb = (slim(gold, nav["gmap_embeds"].cpu(), "gmap_embeds") - gold["gmap_embeds"]).abs()
    lg, lr = nav["global_logits"].cpu(), gold["global_logits"]
    assert torch.equal(torch.isinf(lg), torch.isinf(lr)), "-inf pattern differs"
    fin = ~torch.isinf(lr)
    e_log = (lg[fin] - lr[fin]).abs()
    inside = (e_log <= 1e-4 + 1e-3 * lr[fin].abs()).float().mean().item()
    top2 = lr.masked_fill(~fin, -1e9).topk(2, dim=1).values
    _report(case=name, txt_max=e_txt_valid.max().item(), pano_max=e_pano.max().item(), embed_max=e_emb.max().item(),
            logit_max=e_log.max().item(), logit_mean=e_log.mean().item(), frac_in_northstar_band=inside,
            min_top2_gap=(top2[:, 0] - top2[:, 1]).min().item())
    assert torch.equal(lg.argmax(1), lr.argmax(1)), "node selection differs from the reference"
    gap = (top2[:, 0] - top2[:, 1]).min().item()
    assert gap >= NEAR_TIE_FACTOR * e_log.max().item(), (
        f"near tie: the fixture's smallest top-2 logit gap {gap:.4g} is within {NEAR_TIE_FACTOR}x of the measured logit error "
        f"{e_log.max().item():.4g}: bit-exact node selection would rest on luck")
    assert e_pano.max() < MAX_ABS_EMBED, e_pano.max()
    assert e_emb.max() < MAX_ABS_EMBED, e_emb.max()
    assert e_log.max() < MAX_ABS_LOGIT, e_log.max()
    assert e_txt_valid.max() < MAX_ABS_EMBED, e_txt_valid.max()


def test_forward_c3_shape_vs_oracle_properties():
    """Full BASELINE size (B=64, V=12, N=80, L=200): size-independent properties — finite outputs, exact -inf
    pattern, permutation equivariance over the batch axis (each episode is independent)."""
    from etpnav_b200.config import PlannerConfig
    from etpnav_b200.synth import make_inputs, make_weights
    cfg = PlannerConfig(vocab_size=2048, num_l_layers=1)
    sd = make_weights(cfg, seed=5)
    m = _model(cfg, sd)
    inp = _cuda(make_inputs(cfg, 64, 12, 80, 200, seed=5, ragged=True))
    args = lambda d: (d["txt_embeds"], d["txt_masks"], None, d["gmap_step_ids"], d["gmap_img_fts"], d["gmap_pos_fts"],
                      d["gmap_masks"], d["gmap_visited_masks"], d["gmap_pair_dists"])
    with torch.no_grad():
        nav = m.forward_navigation(*args(inp))
        pano, pm = m.forward_panorama(inp["rgb_fts"], inp["dep_fts"], inp["loc_fts"], inp["nav_types"], inp["view_lens"])
        perm = torch.randperm(64, device="cuda")
        pin = {k: (v[perm] if isinstance(v, torch.Tensor) else v) for k, v in inp.items()}
        nav_p = m.forward_navigation(*args(pin))
    lg = nav["global_logits"]
    dead = inp["gmap_visited_masks"] | ~inp["gmap_masks"]
    assert torch.equal(torch.isinf(lg), dead)
    assert torch.isfinite(nav["gmap_embeds"]).all() and torch.isfinite(pano).all()
    assert torch.equal(nav_p["global_logits"], lg[perm]), "batch permutation changed the logits"
    assert torch.equal(nav_p["gmap_embeds"], nav["gmap_embeds"][perm])


def test_prefetcher_matches_direct_copy():
    """HostInputPrefetcher hands out, step after step, exactly the tensors that were submitted (two slots in flight)."""
    from etpnav_b200.pipeline import HostInputPrefetcher
    dev = torch.device("cuda", 0)
    pf = HostInputPrefetcher(dev)
    g = torch.Generator().manual_seed(3)
    hosts = [{"a": torch.randn(257, 33, generator=g).pin_memory(), "ids": torch.randint(0, 9, (64, 7), generator=g).pin_memory(),
              "tag": i} for i in range(5)]
    pf.submit(hosts[0])
    for i in range(5):
        d = pf.get()
        if i + 1 < 5:
            pf.submit(hosts[i + 1])
        # a long-ish kernel on the compute stream so the next copy really overlaps a consumer of this slot
        acc = d["a"].clone()
        for _ in range(20):
            acc = acc * 1.0001 + d["a"]
        assert d["tag"] == i
        torch.cuda.synchronize()
        assert torch.equal(d["a"].cpu(), hosts[i]["a"]) and torch.equal(d["ids"].cpu(), hosts[i]["ids"])
    with pytest.raises(RuntimeError):
        pf.get()
