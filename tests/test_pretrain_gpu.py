"""GPU: the pre-training twin (etpnav_b200/pretrain.py: B200TextPathCMT / B200PreTraining, SURVEY.md §8f N2) through
the C ABI against the fixtures minted from the UNMODIFIED reference pre-training model (tests/golden/pretrain,
oracle/make_golden_pretrain.py) and against the fp32 oracle port's autograd.  Same numerical contract as the
navigation model's tests (tests/test_planner_gpu.py, tests/test_backward_gpu.py): bf16 GEMM operands, fp32 everything
else; bit-exact -inf pattern and node selection, absolute envelopes for the embeddings / logits, relative L2 for
gradients; measured values are appended to gpurun_out/parity_report.jsonl."""
import json
import os

import numpy as np
import pytest
import torch

from tests.common import no_dropout
from tests.test_oracle_pretrain import grad_sig, load, names, slim

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600)]
MAX_ABS_EMBED, MAX_ABS_LOGIT, MAX_ABS_SCORE = 6e-2, 4e-2, 6e-2
REL_L2_ACT, REL_NORM_PARAM = 8e-2, 1e-1
REPORT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out", "parity_report.jsonl")


def _report(**kw):
    os.makedirs(os.path.dirname(REPORT), exist_ok=True)
    with open(REPORT, "a") as f:
        f.write(json.dumps(kw) + "\n")


def _cuda(b):
    return {k: (v.cuda() if isinstance(v, torch.Tensor) else v) for k, v in b.items()}


def _model(cfg, sd, train=False):
    from etpnav_b200.pretrain import B200PreTraining
    from oracle.ref_import import ref_key
    m = B200PreTraining(cfg, device="cuda")
    ref_sd = {ref_key(k): v for k, v in sd.items()}
    ref_sd["mlm_head.predictions.decoder.weight"] = ref_sd["bert.embeddings.word_embeddings.weight"]  # tied alias
    m.load_state_dict(ref_sd, strict=True)
    assert set(m.state_dict().keys()) == set(ref_sd.keys())
    return m.train() if train else m.eval()


def _twin_args(b):
    return (b["txt_ids"], b["txt_lens"], b["traj_view_img_fts"], b["traj_view_dep_fts"], b["traj_obj_img_fts"],
            b["traj_loc_fts"], b["traj_nav_types"], b["traj_step_lens"], b["traj_vp_view_lens"], b["traj_vp_obj_lens"],
            b["traj_vpids"], b["traj_cand_vpids"], b["gmap_lens"], b["gmap_step_ids"], b["gmap_pos_fts"],
            b["gmap_pair_dists"], b["gmap_vpids"])


def test_segment_gather_fwd_bwd():
    """etp_segment_gather against the dense product with the same sparse matrix (fp32; sums of <= a few dozen terms)."""
    from etpnav_b200 import lib
    from etpnav_b200.pretrain import Csr, segment_gather
    lib.require_device()
    rng = np.random.default_rng(0)
    R, S, W = 300, 77, 768
    counts = rng.integers(0, 9, S)
    counts[3] = 0
    counts[10] = 40
    ptr = np.zeros(S + 1, dtype=np.int32)
    np.cumsum(counts, out=ptr[1:])
    idx = rng.integers(0, R, ptr[-1]).astype(np.int32)
    wt = rng.random(ptr[-1]).astype(np.float32)
    csr = Csr(ptr, idx, wt, R)
    A = torch.zeros(S, R, dtype=torch.float64)
    for s in range(S):
        for k in range(ptr[s], ptr[s + 1]):
            A[s, idx[k]] += float(wt[k])
    src = torch.randn(R, W, device="cuda", requires_grad=True)
    out = segment_gather(src, csr)
    dout = torch.randn(S, W, device="cuda")
    out.backward(dout)
    torch.cuda.synchronize()
    torch.testing.assert_close(out.detach().cpu().double(), A @ src.detach().cpu().double(), rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(src.grad.cpu().double(), A.t() @ dout.cpu().double(), rtol=1e-5, atol=1e-5)
    assert out[3].abs().max().item() == 0.0   # empty segment -> zeros


@pytest.mark.parametrize("name", names())
def test_twin_forward_matches_reference_fixture(name):
    gold, cfg, sd, b = load(name)
    m = _model(cfg, sd)
    d = _cuda(b)
    with torch.no_grad():
        gmap = m.bert(*_twin_args(d))
        mlm_txt = m.bert.forward_mlm(*_twin_args(d))
        logits, labels = m(d, "sap", compute_loss=False)
        scores = m(d, "mlm", compute_loss=False)
        sap_loss, mlm_loss = m(d, "sap"), m(d, "mlm")
    torch.cuda.synchronize()
    lg, lr = logits.cpu(), gold["sap_logits"]
    assert torch.equal(torch.isinf(lg), torch.isinf(lr)), "-inf pattern differs"
    fin = ~torch.isinf(lr)
    gm = (torch.arange(gmap.shape[1])[None] < b["gmap_lens"][:, None])[..., None]
    tm = (torch.arange(b["txt_ids"].shape[1])[None] < b["txt_lens"][:, None])[..., None]
    e_g = (slim(gold, (gmap.cpu() * gm)) - slim(gold, gm.float()) * gold["gmap_embeds"]).abs().max().item()
    e_t = (slim(gold, (mlm_txt.cpu() * tm)) - slim(gold, tm.float()) * gold["mlm_txt_embeds"]).abs().max().item()
    e_l = (lg[fin] - lr[fin]).abs().max().item()
    e_s = (slim(gold, scores.cpu()) - gold["mlm_scores"]).abs().max().item()
    e_sl = (sap_loss.cpu() - gold["sap_loss"]).abs().max().item()
    e_ml = (mlm_loss.cpu() - gold["mlm_loss"]).abs().max().item()
    _report(case=name, kind="pretrain_forward", gmap_max=e_g, mlm_txt_max=e_t, sap_logit_max=e_l, mlm_score_max=e_s,
            sap_loss_max=e_sl, mlm_loss_max=e_ml)
    assert torch.equal(lg.argmax(1), lr.argmax(1)), "node selection differs from the reference"
    assert e_g < MAX_ABS_EMBED and e_t < MAX_ABS_EMBED, (e_g, e_t)
    assert e_l < MAX_ABS_LOGIT, e_l
    assert e_s < MAX_ABS_SCORE, e_s
    assert e_sl < 5e-2 and e_ml < 1e-1, (e_sl, e_ml)


@pytest.mark.parametrize("name", names())
def test_twin_backward_matches_reference_fixture(name):
    """loss = mean(mlm) + mean(sap) as in the fixture: gradient w.r.t. the view features (through lang2visn / the map
    encoder, the segment gather and the pano encoder) and every parameter-gradient signature."""
    gold, cfg, sd, b = load(name)
    no_dropout(cfg)
    m = _model(cfg, sd, train=True)
    d = _cuda(b)
    d["traj_view_img_fts"] = d["traj_view_img_fts"].clone().requires_grad_(True)
    loss = m(d, "mlm").mean() + m(d, "sap").mean()
    loss.backward()
    torch.cuda.synchronize()
    want = gold["mlm_loss"].mean() + gold["sap_loss"].mean()
    rep = {"case": name, "kind": "pretrain_backward", "loss_err": abs(loss.item() - want.item())}
    assert rep["loss_err"] < 2e-2 * max(1.0, abs(want.item())), rep
    g = slim(gold, d["traj_view_img_fts"].grad.cpu())
    rep["d_view_img"] = ((g - gold["grad_traj_view_img_fts"]).norm() / gold["grad_traj_view_img_fts"].norm()).item()
    worst = ("", 0.0)
    for k, sig in gold["param_grad_sig"].items():
        if k == "mlm_head.predictions.decoder.weight":
            continue
        p = m.bert._pmap[k]
        assert p.grad is not None, k
        got = grad_sig(p.grad.cpu())
        ref_norm = float(sig[1])
        if ref_norm < 1e-6:
            assert float(got[1]) < 1e-2, (k, got)
            continue
        e = abs(float(got[1]) - ref_norm) / ref_norm
        e8 = float((got[2:] - sig[2:]).abs().max()) / max(float(sig[2:].abs().max()), 1e-3 * ref_norm)
        if max(e, 0.2 * e8) > worst[1]:
            worst = (k, max(e, 0.2 * e8))
        rep.setdefault("fails", [])
        # e8 looks at 8 single elements: on the 3-episode fixture they are a few bf16 roundings of a handful of token
        # products (measured on B200: up to 0.31 there with the norm within 0.2 %; 0.09 on pt_mid)
        if not (e < REL_NORM_PARAM and e8 < 0.45):
            rep["fails"].append((k, e, e8))
    rep["worst_param"] = worst
    _report(**rep)
    assert rep["d_view_img"] < REL_L2_ACT, rep
    assert not rep["fails"], rep["fails"][:8]


def test_pretrain_trainer_matches_autograd_and_learns():
    """PretrainTrainer accumulates every gradient straight into the flat buffer: it must equal what autograd collects
    parameter by parameter for the same batch (dropout off), and a few iterations on one batch must reduce both losses."""
    from etpnav_b200.pretrain import PretrainTrainer
    gold, cfg, sd, b = load("pt_small")
    no_dropout(cfg)
    d = _cuda(b)
    m = _model(cfg, sd, train=True)
    m(d, "mlm").mean().backward()
    ref = {k: p.grad.clone() for k, p in m.bert._pmap.items() if p.grad is not None}
    m2 = _model(cfg, sd, train=True)
    tr = PretrainTrainer(m2, lr=0.0, weight_decay=0.0)
    first = {t: tr.step(d, t).item() for t in ("mlm", "sap")}
    tr.m._direct_grad.zero_()
    m2(d, "mlm").mean().backward()
    torch.cuda.synchronize()
    lay = m2.bert.layout
    for k, g in ref.items():
        off, numel, shape = lay.entries[k]
        got = tr.m._direct_grad[off:off + numel].view(shape)
        denom = g.norm().clamp_min(1e-12)
        assert ((got - g).norm() / denom).item() < 1e-3, k     # same kernels, same order: fp32 atomics noise only
    tr.lr = 1e-4
    for _ in range(8):
        for t in ("mlm", "sap"):
            last_t = tr.step(d, t).item()
            first.setdefault("last_" + t, 0.0)
            first["last_" + t] = last_t
    torch.cuda.synchronize()
    _report(kind="pretrain_trainer", **first)
    assert first["last_mlm"] < first["mlm"] and first["last_sap"] < first["sap"], first
