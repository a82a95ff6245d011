"""CPU: the oracle restatement (oracle/planner_port.py) against the golden fixtures minted from
the unmodified reference (oracle/make_golden.py), in fp32 and, on one case, in fp64."""
import os

import pytest
import torch

from oracle import planner_port as P
from oracle.make_golden import FP64_CASE
from tests.common import GOLDEN_DIR, golden_loss, golden_names, grad_sig, load_case, slim


@pytest.mark.parametrize("name", golden_names())
def test_port_matches_golden_forward_and_backward(name):
    gold, cfg, sd, inp = load_case(name)
    for k, v in gold["input_sig"].items():  # the seeded generators reproduce the fixture's inputs
        assert torch.allclose(grad_sig(inp[k].float()), v, rtol=1e-5, atol=1e-5), k
    sd = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    txt = P.forward_txt(sd, cfg, inp["txt_ids"], inp["txt_masks"])
    assert torch.allclose(slim(gold, txt, "txt_embeds"), gold["txt_embeds"], rtol=1e-4, atol=2e-5)
    leaves = {k: inp[k].clone().requires_grad_(True) for k in ("rgb_fts", "dep_fts", "gmap_img_fts")}
    txt_leaf = txt.detach().clone().requires_grad_(True)
    pano, pm = P.forward_panorama(sd, cfg, leaves["rgb_fts"], leaves["dep_fts"], inp["loc_fts"],
                                  inp["nav_types"], inp["view_lens"])
    nav = P.forward_navigation(sd, cfg, txt_leaf, inp["txt_masks"], None, inp["gmap_step_ids"],
                               leaves["gmap_img_fts"], inp["gmap_pos_fts"], inp["gmap_masks"],
                               inp["gmap_visited_masks"], inp["gmap_pair_dists"])
    assert torch.equal(pm, gold["pano_masks"])
    assert torch.allclose(slim(gold, pano, "pano_embeds"), gold["pano_embeds"], rtol=1e-4, atol=2e-5)
    assert torch.allclose(slim(gold, nav["gmap_embeds"], "gmap_embeds"), gold["gmap_embeds"], rtol=1e-4, atol=2e-5)
    lg, lr = nav["global_logits"], gold["global_logits"]
    assert torch.equal(torch.isinf(lg), torch.isinf(lr))
    fin = ~torch.isinf(lr)
    assert torch.allclose(lg[fin], lr[fin], rtol=1e-4, atol=1e-5)
    assert torch.equal(lg.argmax(1), lr.argmax(1))  # node selection is bit-exact
    loss = golden_loss(gold, pano, pm, nav["gmap_embeds"], lg, inp)
    assert torch.allclose(loss, gold["loss"], rtol=1e-5, atol=1e-4)
    loss.backward()
    assert torch.allclose(slim(gold, txt_leaf.grad, "grad_txt_embeds"), gold["grad_txt_embeds"], rtol=1e-3, atol=1e-6)
    for k, v in leaves.items():
        if "grad_" + k in gold:
            assert torch.allclose(slim(gold, v.grad, "grad_" + k), gold["grad_" + k], rtol=1e-3, atol=1e-6), k
    for k, sig in gold["param_grad_sig"].items():
        if k.startswith("lang_encoder") or k.startswith("embeddings.word") \
                or k.startswith("embeddings.position") or k.startswith("embeddings.LayerNorm"):
            continue  # forward_txt output was detached into txt_leaf in the fixture too
        got = grad_sig(sd[k].grad)
        tol = 1e-4 * float(sig[1]) + 2e-6  # sprel bias grad is analytically 0 (softmax shift invariance)
        assert torch.allclose(got, sig, rtol=2e-3, atol=tol), (k, got, sig)


def test_port_matches_reference_fp64():
    """The port in fp64 against the unmodified reference's own fp64 outputs (tests/golden/fp64,
    oracle/make_golden.py:run_fp64).  The port's nav step consumes the port's txt_embeds, which the first assertion
    pins to the reference's."""
    gold, cfg, sd, inp = load_case(FP64_CASE)
    ref = torch.load(os.path.join(GOLDEN_DIR, "fp64", FP64_CASE + ".pt"), weights_only=False)
    cols = ref["cols"]
    sd64 = {k: v.double() for k, v in sd.items()}
    f = lambda t: t.double() if t.dtype.is_floating_point else t
    i64 = {k: f(v) if isinstance(v, torch.Tensor) else v for k, v in inp.items()}
    with torch.no_grad():
        t_port = P.forward_txt(sd64, cfg, i64["txt_ids"], i64["txt_masks"])
        assert (ref["txt_embeds"] - t_port[..., cols]).abs().max() < 1e-11
        p_port, m_port = P.forward_panorama(sd64, cfg, i64["rgb_fts"], i64["dep_fts"], i64["loc_fts"],
                                            i64["nav_types"], i64["view_lens"])
        assert torch.equal(ref["pano_masks"], m_port) and (ref["pano_embeds"] - p_port[..., cols]).abs().max() < 1e-11
        args = (t_port, i64["txt_masks"], None, i64["gmap_step_ids"], i64["gmap_img_fts"], i64["gmap_pos_fts"],
                i64["gmap_masks"], i64["gmap_visited_masks"], i64["gmap_pair_dists"])
        n_port = P.forward_navigation(sd64, cfg, *args)
        assert (ref["gmap_embeds"] - n_port["gmap_embeds"][..., cols]).abs().max() < 1e-11
        fin = ~torch.isinf(ref["global_logits"])
        assert torch.equal(fin, ~torch.isinf(n_port["global_logits"]))
        assert (ref["global_logits"][fin] - n_port["global_logits"][fin]).abs().max() < 1e-11


def test_port_full_gradients_match_reference_sketches():
    """The port's FULL parameter gradients on c1_bert against the sketches of the unmodified reference's gradients
    (tests/golden/grads: all row sums, all column sums, 64 sampled entries per matrix, full 1-D tensors)."""
    from oracle.make_golden_grads import TEXT_PREFIXES
    from tests.common import GOLDEN_GRADS_DIR
    gold, cfg, sd, inp = load_case("c1_bert")
    sk = torch.load(os.path.join(GOLDEN_GRADS_DIR, "c1_bert.pt"), weights_only=False)
    sd = {k: (v.clone().requires_grad_(True) if not k.startswith(TEXT_PREFIXES) else v) for k, v in sd.items()}
    txt = gold["txt_embeds"]
    pano, pm = P.forward_panorama(sd, cfg, inp["rgb_fts"], inp["dep_fts"], inp["loc_fts"], inp["nav_types"], inp["view_lens"])
    nav = P.forward_navigation(sd, cfg, txt, inp["txt_masks"], None, inp["gmap_step_ids"], inp["gmap_img_fts"],
                               inp["gmap_pos_fts"], inp["gmap_masks"], inp["gmap_visited_masks"], inp["gmap_pair_dists"])
    loss = golden_loss(gold, pano, pm, nav["gmap_embeds"], nav["global_logits"], inp)
    assert torch.allclose(loss, sk["loss"], rtol=1e-5, atol=1e-4)
    loss.backward()
    assert len(sk["sketch"]) >= 150
    for k, ref in sk["sketch"].items():
        g = sd[k].grad
        assert g is not None, k
        if "full" in ref:
            assert torch.allclose(g, ref["full"], rtol=2e-3, atol=1e-5 * float(ref["full"].abs().max()) + 2e-7), k
            continue
        g2 = g.reshape(g.shape[0], -1)
        big = float(g2.abs().max()) * g2.shape[1] ** 0.5
        assert torch.allclose(g2.flatten()[ref["idx"]], ref["vals"], rtol=2e-3, atol=1e-5 * float(g2.abs().max()) + 2e-7), k
        assert torch.allclose(g2.double().sum(1).float(), ref["row_sum"], rtol=2e-3, atol=2e-5 * big + 2e-7), k
        assert torch.allclose(g2.double().sum(0).float(), ref["col_sum"], rtol=2e-3, atol=2e-5 * float(g2.abs().max()) * g2.shape[0] ** 0.5 + 2e-7), k
