"""GPU: the high-precision inference mode (``B200Planner.set_precision("high")``: split-bf16 x3 GEMMs on tcgen05 +
fp32 attention) meets BASELINE.json's north_star band — rtol 1e-3 / atol 1e-4 on every node logit and every embedding,
node selection and the -inf pattern bit-exact — against the golden fixtures minted from the UNMODIFIED reference in
fp32 (tests/golden, oracle/make_golden.py).  That is the reference's own eval / inference arithmetic
(ss_trainer_ETP.py:513-756 runs without autocast).  The tolerance is the north_star's, written here: RTOL, ATOL."""
import json
import os

import pytest
import torch

from tests.common import golden_names, load_case, slim

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600)]

RTOL, ATOL = 1e-3, 1e-4
REPORT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out", "parity_report_hp.jsonl")


def _report(**kw):
    os.makedirs(os.path.dirname(REPORT), exist_ok=True)
    with open(REPORT, "a") as f:
        f.write(json.dumps(kw) + "\n")


def _in_band(x, ref):
    return (x - ref).abs() <= ATOL + RTOL * ref.abs()


def test_split3_gemm_is_fp32_accurate():
    """D = A.B^T through etp_split3 + the unchanged tcgen05 GEMM with K' = 3K, against float64."""
    from etpnav_b200 import lib as L
    g = torch.Generator(device="cuda").manual_seed(1)
    for M, N, K in [(300, 768, 768), (129, 256, 3072), (64, 2304, 128)]:
        A = torch.randn(M, K, device="cuda", generator=g)
        B = torch.randn(N, K, device="cuda", generator=g) * 0.05
        bias = torch.randn(N, device="cuda", generator=g)
        out = torch.empty(M, N, device="cuda")
        L.gemm(L.split3(A, 0), L.split3(B, 1), bias=bias, out_f32=out)
        ref = (A.double() @ B.double().t() + bias.double())
        err = (out.double() - ref).abs().max().item()
        scale = ref.abs().max().item()
        assert err < 2e-5 * scale, (M, N, K, err, scale)
        # the same product with plain bf16 operands is ~2^8 times worse: the split is doing the work
        out16 = torch.empty(M, N, device="cuda")
        L.gemm(A.bfloat16(), B.bfloat16(), bias=bias, out_f32=out16)
        assert (out16.double() - ref).abs().max().item() > 20 * err


@pytest.mark.parametrize("B,Sq,Sk,pair,ninf", [(3, 80, 200, False, False), (2, 80, 80, True, False), (4, 12, 12, False, True),
                                               (1, 130, 513, True, False)])
def test_attention_f32_matches_float64(B, Sq, Sk, pair, ninf):
    from etpnav_b200 import lib as L
    g = torch.Generator(device="cuda").manual_seed(2)
    h = 12
    q = torch.randn(B * Sq, 768, device="cuda", generator=g)
    kv = torch.randn(B * Sk, 1536, device="cuda", generator=g)
    valid = torch.rand(B, Sk, device="cuda", generator=g) > 0.3
    valid[:, 0] = True
    pd = torch.rand(B, Sq, Sk, device="cuda", generator=g) if pair else None
    out = torch.empty(B * Sq, 768, device="cuda")
    mv = float("-inf") if ninf else -10000.0
    L.attention_f32_fwd(q, kv[:, :768], kv[:, 768:], out, B=B, heads=h, Sq=Sq, Sk=Sk, key_valid=valid.view(torch.uint8),
                        mask_value=mv, pair=pd, pair_w=0.7, pair_b=-0.2)
    qh = q.double().view(B, Sq, h, 64).permute(0, 2, 1, 3)
    kh = kv[:, :768].double().view(B, Sk, h, 64).permute(0, 2, 1, 3)
    vh = kv[:, 768:].double().view(B, Sk, h, 64).permute(0, 2, 1, 3)
    s = qh @ kh.transpose(-1, -2) * 0.125
    s = s + torch.where(valid, 0.0, mv).double()[:, None, None, :]
    if pair:
        s = s + (0.7 * pd.double() - 0.2)[:, None]
    ref = (torch.softmax(s, -1) @ vh).permute(0, 2, 1, 3).reshape(B * Sq, 768)
    assert (out.double() - ref).abs().max().item() < 2e-5


@pytest.mark.parametrize("name", golden_names())
def test_high_precision_forward_in_northstar_band(name):
    from etpnav_b200.planner import B200Planner
    gold, cfg, sd, inp = load_case(name)
    m = B200Planner(cfg, device="cuda")
    m.load_state_dict(sd, strict=True)
    m.eval().set_precision("high")
    d = {k: (v.cuda() if isinstance(v, torch.Tensor) else v) for k, v in inp.items()}
    with torch.no_grad():
        txt = m.forward_txt(d["txt_ids"], d["txt_masks"])
        pano, pmask = m.forward_panorama(d["rgb_fts"], d["dep_fts"], d["loc_fts"], d["nav_types"], d["view_lens"])
        # end to end: the navigation step consumes THIS mode's own txt_embeds (no reference tensor is fed back in)
        nav = m.forward_navigation(txt, d["txt_masks"], None, d["gmap_step_ids"], d["gmap_img_fts"], d["gmap_pos_fts"],
                                   d["gmap_masks"], d["gmap_visited_masks"], d["gmap_pair_dists"])
    torch.cuda.synchronize()
    lg, lr = nav["global_logits"].cpu(), gold["global_logits"]
    assert torch.equal(torch.isinf(lg), torch.isinf(lr)), "-inf pattern differs"
    fin = ~torch.isinf(lr)
    ok_log = _in_band(lg[fin], lr[fin])
    e_log = (lg[fin] - lr[fin]).abs()
    checks = {"txt": (slim(gold, txt.cpu(), "txt_embeds"), gold["txt_embeds"]),
              "pano": (slim(gold, pano.cpu(), "pano_embeds"), gold["pano_embeds"]),
              "gmap": (slim(gold, nav["gmap_embeds"].cpu(), "gmap_embeds"), gold["gmap_embeds"])}
    rep = {"case": name, "mode": "high", "logit_max": e_log.max().item(), "frac_in_northstar_band": ok_log.float().mean().item()}
    for k, (x, r) in checks.items():
        rep[k + "_max"] = (x - r).abs().max().item()
        rep[k + "_frac_in_band"] = _in_band(x, r).float().mean().item()
    top2 = lr.masked_fill(~fin, -1e9).topk(2, dim=1).values
    rep["min_top2_gap"] = (top2[:, 0] - top2[:, 1]).min().item()
    _report(**rep)
    assert torch.equal(pmask.cpu(), gold["pano_masks"])
    assert torch.equal(lg.argmax(1), lr.argmax(1)), "node selection differs from the reference"
    assert ok_log.all(), f"logits outside rtol {RTOL} / atol {ATOL}: max |d| {e_log.max().item()}"
    for k, (x, r) in checks.items():
        assert _in_band(x, r).all(), f"{k} embeddings outside the band: max |d| {(x - r).abs().max().item()}"
    # node selection is safe by construction in this mode: the top-2 gap dwarfs the error
    assert rep["min_top2_gap"] > 20 * rep["logit_max"]


def test_high_precision_is_inference_only():
    from etpnav_b200 import lib as L
    from etpnav_b200.config import PlannerConfig
    from etpnav_b200.planner import B200Planner
    from etpnav_b200.synth import make_inputs
    cfg = PlannerConfig(vocab_size=2048, num_l_layers=1, num_x_layers=1)
    m = B200Planner(cfg, device="cuda").train().set_precision("high")
    d = {k: (v.cuda() if isinstance(v, torch.Tensor) else v) for k, v in make_inputs(cfg, 2, 12, 8, 16, seed=0, ragged=False).items()}
    with pytest.raises(L.EtpError):
        m.forward_panorama(d["rgb_fts"], d["dep_fts"], d["loc_fts"], d["nav_types"], d["view_lens"])
    # weights changed through torch: the hi|hi|lo image follows (version key), like the bf16 image
    m.eval()
    with torch.no_grad():
        a = m.forward_panorama(d["rgb_fts"], d["dep_fts"], d["loc_fts"], d["nav_types"], d["view_lens"])[0].clone()
        m._pmap["img_embeddings.pano_encoder.layers.0.linear2.weight"].mul_(1.5)
        b = m.forward_panorama(d["rgb_fts"], d["dep_fts"], d["loc_fts"], d["nav_types"], d["view_lens"])[0]
    assert (a - b).abs().max().item() > 1e-3
