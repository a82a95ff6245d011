"""CPU: the pre-training oracle port (oracle/pretrain_port.py) reproduces the fixtures minted from the UNMODIFIED
reference (oracle/make_golden_pretrain.py), and the host-side index form of _aggregate_gmap_features
(etpnav_b200/pretrain.py:build_gmap_csr) equals the reference's dictionary loops."""
import glob
import os

import numpy as np
import pytest
import torch

from etpnav_b200.config import PlannerConfig
from etpnav_b200.synth import make_traj_batch, make_weights
from oracle import pretrain_port as PP

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "pretrain")


def names():
    return sorted(os.path.splitext(os.path.basename(p))[0] for p in glob.glob(os.path.join(GOLD, "*.pt")))


def load(name):
    gold = torch.load(os.path.join(GOLD, name + ".pt"), weights_only=False)
    c = gold["case"]
    cfg = PlannerConfig(**c["cfg"])
    sd = make_weights(cfg, seed=c["wseed"])
    b = make_traj_batch(cfg, c["B"], c["T"], c["V"], c["L"], seed=c["iseed"], ghosts=c["ghosts"])
    return gold, cfg, sd, b


def slim(gold, t, dim=1):
    s = gold["case"].get("slim")
    if not s:
        return t
    return t[:, ::s]


def grad_sig(t):
    t = t.detach().double().flatten()
    return torch.cat([t.sum()[None], t.norm()[None], t[:8]]).float()


@pytest.mark.parametrize("name", names())
def test_port_matches_reference_fixture(name):
    gold, cfg, sd, b = load(name)
    sd = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    b = dict(b)
    b["traj_view_img_fts"] = b["traj_view_img_fts"].clone().requires_grad_(True)
    nav = PP.forward_gmap(sd, cfg, b)
    tol = dict(rtol=1e-4, atol=2e-5)
    torch.testing.assert_close(slim(gold, nav["gmap_embeds"].detach()), gold["gmap_embeds"], **tol)
    assert torch.equal(torch.isinf(nav["global_logits"]), torch.isinf(gold["sap_logits"]))
    fin = ~torch.isinf(gold["sap_logits"])
    torch.testing.assert_close(nav["global_logits"].detach()[fin], gold["sap_logits"][fin], **tol)
    torch.testing.assert_close(slim(gold, PP.forward_mlm(sd, cfg, b).detach()), gold["mlm_txt_embeds"], **tol)
    torch.testing.assert_close(slim(gold, PP.task_mlm(sd, cfg, b, compute_loss=False).detach()), gold["mlm_scores"],
                               rtol=1e-4, atol=1e-4)
    sap, mlm = PP.task_sap(sd, cfg, b), PP.task_mlm(sd, cfg, b)
    torch.testing.assert_close(sap.detach(), gold["sap_loss"], **tol)
    torch.testing.assert_close(mlm.detach(), gold["mlm_loss"], rtol=1e-4, atol=1e-4)
    (mlm.mean() + sap.mean()).backward()
    torch.testing.assert_close(slim(gold, b["traj_view_img_fts"].grad), gold["grad_traj_view_img_fts"], rtol=2e-3, atol=1e-7)
    checked = 0
    for k, sig in gold["param_grad_sig"].items():
        if k == "mlm_head.predictions.decoder.weight":
            continue  # tied: its gradient is accumulated into embeddings.word_embeddings.weight
        g = sd[k].grad
        assert g is not None, k
        # the first entry is a sum with heavy cancellation: absolute tolerance relative to the gradient's norm
        torch.testing.assert_close(grad_sig(g), sig, rtol=5e-3, atol=2e-6 + 1e-4 * float(sig[1]),
                                   msg=lambda m, k=k: f"{k}: {m}")
        checked += 1
    assert checked > 60


@pytest.mark.parametrize("seed", [0, 1, 2, 3])
def test_csr_equals_reference_dictionary_loops(seed):
    from etpnav_b200.pretrain import build_gmap_csr
    cfg = PlannerConfig(vocab_size=2048)
    b = make_traj_batch(cfg, 5, 5, 9, 12, seed=seed, ghosts=4 + seed)
    g = torch.Generator().manual_seed(seed)
    S, V, H = b["traj_view_img_fts"].shape[0], b["traj_view_img_fts"].shape[1], 8
    emb = torch.randn(S, V, H, generator=g, dtype=torch.float64)
    se = torch.split(emb, b["traj_step_lens"], 0)
    sl = torch.split(b["traj_vp_view_lens"], b["traj_step_lens"], 0)
    want = PP.aggregate_gmap_features(se, sl, b["traj_vpids"], b["traj_cand_vpids"], b["gmap_vpids"])
    csr, n_max = build_gmap_csr(b["traj_step_lens"], b["traj_vp_view_lens"].tolist(), b["traj_vpids"],
                                b["traj_cand_vpids"], b["gmap_vpids"], V)
    assert n_max == want.shape[1] == b["gmap_step_ids"].shape[1]
    A = np.zeros((csr.num_segments, csr.num_src))
    for s in range(csr.num_segments):
        for k in range(csr.seg_ptr[s], csr.seg_ptr[s + 1]):
            A[s, csr.index[k]] += csr.weight[k]
    got = torch.from_numpy(A) @ emb.reshape(S * V, H)
    torch.testing.assert_close(got.view(want.shape), want, rtol=1e-6, atol=1e-7)  # fp32 weights 1/len
    # the transposed structure is the adjoint
    t = csr.transposed()
    At = np.zeros((t.num_segments, t.num_src))
    for s in range(t.num_segments):
        for k in range(t.seg_ptr[s], t.seg_ptr[s + 1]):
            At[s, t.index[k]] += t.weight[k]
    assert np.array_equal(At, A.T)


def test_pretraining_state_dict_keys_match_reference_layout():
    """B200PreTraining uses the reference's key layout (bert.*, mlm_head.* with the tied decoder, global_sap_head.*);
    checked against the key list stored by the fixture generator (parameter-gradient signature keys + tied alias)."""
    from etpnav_b200.spec import param_shapes
    gold, cfg, _, _ = load("pt_small")
    mine = set(param_shapes(cfg).keys())
    ref = set(gold["param_grad_sig"].keys()) - {"mlm_head.predictions.decoder.weight"}
    # every parameter that received a gradient in the reference exists here under the same (prefix-stripped) name
    assert ref <= mine, sorted(ref - mine)
    assert {k for k in mine if ".lang_" in k} <= ref
