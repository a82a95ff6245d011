"""GPU: training through the episode-level text K|V handle (``encode_text_kv`` with gradients enabled).

The reference encodes the instruction once per rollout (ss_trainer_ETP.py:801), indexes ``all_txt_embeds[not_done_index]``
at every step (:819-822), sums the steps' losses and runs ONE backward (:504) with weights that do not change in between.
A training handle keeps the rollout's bf16 K|V once; each step's backward adds its dK|dV into the handle's fp32
accumulator through the row map, and one node after the rollout runs the key|value weight gradient and d txt_embeds.
The forward must equal the un-cached step, the gradients must match the un-cached rollout, and the stack the reference
trainer wraps around the planner (DDP, autocast, GradScaler) must keep working."""
import os

import pytest
import torch

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600)]

# K|V weights and the language encoder: the un-cached rollout rounds each step's dK|dV to bf16 before its own weight /
# data gradient GEMM, the handle sums the steps in fp32 and rounds once.  Bound <= 2x the largest relative L2 difference
# measured on a B200 (2.9e-3, DESIGN.md §5a).
KV_REL_TOL = 5e-3
OTHER_REL_TOL = 1e-4
# d b4 of the SAP head = sum of the CE gradient over each row's logits, zero in exact arithmetic: rounding noise only
ZERO_GRADS = ("global_sap_head.net.4.bias",)


def _model(X=2, NL=1, dropout=True, seed=13):
    from etpnav_b200.config import PlannerConfig
    from etpnav_b200.planner import B200Planner
    from etpnav_b200.synth import make_weights
    from tests.common import no_dropout
    cfg = PlannerConfig(vocab_size=2048, num_l_layers=NL, num_x_layers=X)
    if not dropout:
        no_dropout(cfg)
    m = B200Planner(cfg, device="cuda")
    m.load_state_dict(make_weights(cfg, seed=seed), strict=True)
    return cfg, m


def _steps(cfg, B0, Ns, L, seed=60):
    from etpnav_b200.synth import make_inputs
    out = []
    for t, N in enumerate(Ns):
        inp = make_inputs(cfg, B0, 12, N, L, seed=seed + t, ragged=True)
        out.append({k: (v.cuda() if isinstance(v, torch.Tensor) else v) for k, v in inp.items()})
    return out


def _nav(m, txt, d, sel=slice(None), img=None):
    return m.forward_navigation(txt, d["txt_masks"][sel], None, d["gmap_step_ids"][sel],
                                d["gmap_img_fts"][sel] if img is None else img, d["gmap_pos_fts"][sel], d["gmap_masks"][sel],
                                d["gmap_visited_masks"][sel], d["gmap_pair_dists"][sel])


def _rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item()


def _is_text_side(name):
    return (name.startswith("embeddings.") or name.startswith("lang_encoder.")
            or (".visual_attention.att." in name and name.endswith((".key.weight", ".value.weight"))))


def _rollout(m, steps, sels, handle, txt_leaf=None):
    """forward_txt (or the given leaf) once, then per step panorama -> masked mean into a map node -> navigation -> CE(sum)
    on the surviving episodes ``sels[t]`` (a list, as not_done_index), ONE backward.  Returns (loss, param grads,
    d rgb_fts per step, d txt_leaf)."""
    d0 = steps[0]
    m.set_dropout_seed(1234)
    m.zero_grad(set_to_none=True)
    txt = txt_leaf if txt_leaf is not None else m.forward_txt(d0["txt_ids"], d0["txt_masks"])
    src = m.encode_text_kv(txt) if handle else txt
    loss, rgbs = 0.0, []
    for d, sel in zip(steps, sels):
        rgb = d["rgb_fts"][sel].clone().requires_grad_(True)
        rgbs.append(rgb)
        pano, pm = m.forward_panorama(rgb, d["dep_fts"][sel], d["loc_fts"][sel], d["nav_types"][sel], d["view_lens"][sel])
        w = pm.unsqueeze(-1).to(pano.dtype)
        img = d["gmap_img_fts"][sel].clone()
        img[:, 1] = img[:, 1] + (pano * w).sum(1) / w.sum(1)
        out = m.forward_navigation(src[sel], d0["txt_masks"][sel], None, d["gmap_step_ids"][sel], img, d["gmap_pos_fts"][sel],
                                   d["gmap_masks"][sel], d["gmap_visited_masks"][sel], d["gmap_pair_dists"][sel])
        loss = loss + torch.nn.functional.cross_entropy(out["global_logits"], d["labels"][sel], reduction="sum")
    loss.backward()
    torch.cuda.synchronize()
    grads = {n: p.grad.detach().clone() for n, p in m.named_parameters() if p.grad is not None}
    return (loss.item(), grads, [r.grad.detach().clone() for r in rgbs],
            txt_leaf.grad.detach().clone() if txt_leaf is not None else None)


def _compare_rollouts(m, steps, sels, txt_leaf=None):
    """Un-cached vs handle rollout: (worst text-side rel L2, worst other rel L2); asserts the other bound."""
    if txt_leaf is not None:
        txt_leaf.grad = None
    la, ga, ra, ta = _rollout(m, steps, sels, False, txt_leaf)
    if txt_leaf is not None:
        txt_leaf.grad = None
    lb, gb, rb, tb = _rollout(m, steps, sels, True, txt_leaf)
    assert abs(la - lb) <= 1e-5 * abs(la), (la, lb)   # the handle's forward is the un-cached one (last bits at shrunk steps)
    assert ga.keys() == gb.keys()
    text, other = ("", 0.0), ("", 0.0)
    for n in ga:
        if n in ZERO_GRADS:
            assert ga[n].abs().max() < 1e-4 and gb[n].abs().max() < 1e-4, (n, ga[n], gb[n])
            continue
        if ga[n].norm() == 0:
            assert gb[n].norm() == 0, n
            continue
        r = _rel(gb[n], ga[n])
        if _is_text_side(n):
            text = max(text, (n, r), key=lambda t: t[1])
        else:
            other = max(other, (n, r), key=lambda t: t[1])
    for t, (a, b) in enumerate(zip(ra, rb)):
        other = max(other, (f"d rgb_fts[{t}]", _rel(b, a)), key=lambda t: t[1])
    if ta is not None:
        text = max(text, ("d txt_embeds", _rel(tb, ta)), key=lambda t: t[1])
    print("text-side worst rel L2", text, "| other worst rel L2", other)
    assert other[1] <= OTHER_REL_TOL, other
    return text, other


def test_forward_equals_uncached_step_and_tracks_two_shrinks():
    cfg, m = _model(X=3, NL=0)
    m.train()
    (d,) = _steps(cfg, 6, [30], 150)
    txt = d["txt_embeds"].clone().requires_grad_(True)
    kv = m.encode_text_kv(txt)
    assert kv.grad is not None                                   # a training handle
    m.set_dropout_seed(7)
    ref = _nav(m, txt, d)
    m.set_dropout_seed(7)
    got = _nav(m, kv, d)
    assert got["global_logits"].grad_fn is not None
    assert torch.equal(got["global_logits"], ref["global_logits"]) and torch.equal(got["gmap_embeds"], ref["gmap_embeds"])
    keep = [0, 2, 3, 5]
    keep2 = [0, 2, 3]                                            # rows of keep: a second shrink composes with the first
    rows2 = [keep[i] for i in keep2]
    for src_kv, sel in ((kv[keep], keep), (kv[keep][keep2], rows2)):
        m.set_dropout_seed(8)
        r = _nav(m, txt[sel], d, sel)
        m.set_dropout_seed(8)
        g = _nav(m, src_kv, d, sel)
        fin = ~torch.isinf(r["global_logits"])
        assert torch.equal(torch.isinf(g["global_logits"]), ~fin)
        assert (g["global_logits"][fin] - r["global_logits"][fin]).abs().max().item() < 1e-5
        assert (g["gmap_embeds"] - r["gmap_embeds"]).abs().max().item() < 1e-4


def test_rollout_gradients_match_uncached_rollout():
    cfg, m = _model(X=2, NL=1)
    m.train()
    steps = _steps(cfg, 6, [12, 18, 24, 30], 40)                 # the map grows
    sels = [list(range(6)), [0, 1, 3, 5], [0, 3, 5], [0, 3, 5]]  # episodes finish: 6 -> 4 -> 3
    text, _ = _compare_rollouts(m, steps, sels)
    assert text[1] <= KV_REL_TOL, text


def test_cuda_core_backward_with_row_map_and_tiny_shapes():
    # N > 128 nodes: the tensor-core backward takes one 128-row query tile, so the CUDA-core kernels run
    cfg, m = _model(X=1, NL=0, seed=21)
    m.train()
    for Ns, L in (([140, 136], 24), ([10, 12], 12)):             # second: Sq, Sk < 32 (CUDA-core kernels as well)
        steps = _steps(cfg, 3, Ns, L, seed=90 + L)
        txt = steps[0]["txt_embeds"].clone().requires_grad_(True)
        text, _ = _compare_rollouts(m, steps, [[0, 1, 2], [2, 0]], txt_leaf=txt)
        assert text[1] <= KV_REL_TOL, (Ns, L, text)


def test_saved_bytes_and_step_memory():
    from etpnav_b200 import lib as _L
    from etpnav_b200.planner import _declare
    _declare()
    L = _L.lib()
    for B, N, Lt, X in ((64, 80, 200, 6), (3, 17, 40, 1), (6, 30, 150, 3)):
        full = L.etp_nav_saved_bytes(B, N, Lt, X, 1)
        assert full - L.etp_nav_kv_saved_bytes(B, N, Lt, X, 1) == B * Lt * (X * 1536 + 768) * 2
    cfg, m = _model(X=3, NL=0)
    m.train()
    (d,) = _steps(cfg, 6, [30], 150)
    txt = d["txt_embeds"].clone().requires_grad_(True)
    kv = m.encode_text_kv(txt)
    sel = [0, 1, 3, 4, 5]
    B, Lt, X = len(sel), 150, 3

    def growth(src_fn):
        torch.cuda.synchronize()
        a0 = torch.cuda.memory_allocated()
        out = _nav(m, src_fn(), d, sel)
        torch.cuda.synchronize()
        return torch.cuda.memory_allocated() - a0, out

    g_ref, o_ref = growth(lambda: txt[sel])
    g_kv, o_kv = growth(lambda: kv[sel])
    assert g_ref - g_kv >= B * Lt * (X * 1536 + 768) * 2, (g_ref, g_kv)


def test_errors():
    from etpnav_b200 import lib as _L
    cfg, m = _model(X=1, NL=0, dropout=False)
    m.train()
    steps = _steps(cfg, 3, [12], 40)
    d = steps[0]
    with torch.no_grad():
        inf = m.encode_text_kv(d["txt_embeds"])
    assert inf.grad is None
    with pytest.raises(_L.EtpError):
        _nav(m, inf, d)                                          # inference handle where gradients are wanted
    txt = d["txt_embeds"].clone().requires_grad_(True)
    kv = m.encode_text_kv(txt)
    with pytest.raises(ValueError):
        _nav(m, kv[[0, 1]], d)                                   # handle of 2 episodes, step batch of 3
    with torch.no_grad():                                        # a training handle under no_grad = the inference handle
        a, b = _nav(m, kv, d), _nav(m, inf, d)
        assert torch.equal(a["global_logits"], b["global_logits"])
    m.set_precision("high")
    with pytest.raises(_L.EtpError):
        _nav(m, kv, d)                                           # no backward exists for precision="high"
    m.set_precision("bf16")
    out = _nav(m, kv, d)
    out["global_logits"][~torch.isinf(out["global_logits"])].sum().backward()
    assert txt.grad is not None and torch.isfinite(txt.grad).all()
    with pytest.raises(_L.EtpError):
        _nav(m, kv, d)                                           # its backward has run
    with pytest.raises(_L.EtpError), torch.no_grad():
        _nav(m, kv[[0, 1, 2]], d)                                # in any mode, and through an indexed copy


def test_ddp_autocast_gradscaler_rollout_through_the_handle_matches_oracle():
    import torch.distributed as dist
    import torch.nn as nn
    from torch.nn.parallel import DistributedDataParallel as DDP
    from oracle import planner_port as P

    class _Net(nn.Module):
        def __init__(self, planner):
            super().__init__()
            self.vln_bert = planner

        def forward(self, mode=None, **kw):
            if mode == "language":
                return self.vln_bert.forward_txt(kw["txt_ids"], kw["txt_masks"])
            if mode == "text_kv":
                return self.vln_bert.encode_text_kv(kw["txt_embeds"])
            if mode == "panorama":
                return self.vln_bert.forward_panorama(kw["rgb_fts"], kw["dep_fts"], kw["loc_fts"], kw["nav_types"],
                                                      kw["view_lens"])
            return self.vln_bert.forward_navigation(kw["txt_embeds"], kw["txt_masks"], None, kw["gmap_step_ids"],
                                                    kw["gmap_img_fts"], kw["gmap_pos_fts"], kw["gmap_masks"],
                                                    kw["gmap_visited_masks"], kw["gmap_pair_dists"])

    def rollout_loss(call, steps, sels, handle):
        d0 = steps[0]
        txt = call(mode="language", txt_ids=d0["txt_ids"], txt_masks=d0["txt_masks"])
        src = call(mode="text_kv", txt_embeds=txt) if handle else txt
        loss, n = 0.0, 0
        for d, sel in zip(steps, sels):
            pano, pm = call(mode="panorama", rgb_fts=d["rgb_fts"][sel], dep_fts=d["dep_fts"][sel], loc_fts=d["loc_fts"][sel],
                            nav_types=d["nav_types"][sel], view_lens=d["view_lens"][sel])
            w = pm.unsqueeze(-1).to(pano.dtype)
            img = d["gmap_img_fts"][sel].clone()
            img[:, 1] = img[:, 1] + ((pano * w).sum(1) / w.sum(1)).to(img.dtype)
            out = call(mode="navigation", txt_embeds=src[sel], txt_masks=d0["txt_masks"][sel],
                       gmap_step_ids=d["gmap_step_ids"][sel], gmap_img_fts=img, gmap_pos_fts=d["gmap_pos_fts"][sel],
                       gmap_masks=d["gmap_masks"][sel], gmap_visited_masks=d["gmap_visited_masks"][sel],
                       gmap_pair_dists=d["gmap_pair_dists"][sel])
            loss = loss + torch.nn.functional.cross_entropy(out["global_logits"].float(), d["labels"][sel], reduction="sum")
            n += len(sel)
        return loss / n

    from etpnav_b200.synth import make_weights
    torch.cuda.set_device(0)
    own_pg = not dist.is_initialized()
    if own_pg:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29733")
        dist.init_process_group("nccl", rank=0, world_size=1, device_id=torch.device("cuda", 0))
    try:
        cfg, planner = _model(X=2, NL=2, dropout=False, seed=51)
        sd = make_weights(cfg, seed=51)
        net = _Net(planner).train()
        ddp = DDP(net, device_ids=[0], output_device=0, find_unused_parameters=False, broadcast_buffers=False)
        opt = torch.optim.AdamW(ddp.parameters(), lr=1e-3)
        scaler = torch.amp.GradScaler("cuda")
        steps = _steps(cfg, 4, [12, 15, 18], 24)
        sels = [[0, 1, 2, 3], [0, 2, 3], [0, 3]]
        opt.zero_grad()
        with torch.amp.autocast("cuda"):
            loss = rollout_loss(lambda **kw: ddp(**kw), steps, sels, True)
        scaler.scale(loss).backward()
        scaler.unscale_(opt)
        grads = {k: p.grad.detach().clone() for k, p in planner.named_parameters() if p.grad is not None}
        scaler.step(opt)
        scaler.update()
        torch.cuda.synchronize()

        sdc = {k: v.cuda().clone().requires_grad_(True) for k, v in sd.items()}

        def oracle_call(mode=None, **kw):
            if mode == "language":
                return P.forward_txt(sdc, cfg, kw["txt_ids"], kw["txt_masks"])
            if mode == "panorama":
                return P.forward_panorama(sdc, cfg, kw["rgb_fts"], kw["dep_fts"], kw["loc_fts"], kw["nav_types"], kw["view_lens"])
            return P.forward_navigation(sdc, cfg, kw["txt_embeds"], kw["txt_masks"], None, kw["gmap_step_ids"], kw["gmap_img_fts"],
                                        kw["gmap_pos_fts"], kw["gmap_masks"], kw["gmap_visited_masks"], kw["gmap_pair_dists"])
        loss_o = rollout_loss(oracle_call, steps, sels, False)
        loss_o.backward()
        assert abs(loss.item() - loss_o.item()) < 2e-2 * max(1.0, abs(loss_o.item())), (loss.item(), loss_o.item())
        assert len(grads) == len(sd), (len(grads), len(sd))     # every parameter got a gradient (DDP needs that)
        worst = ("", 0.0)
        for k, g in grads.items():
            go = sdc[k].grad
            assert torch.isfinite(g).all(), k
            if go is None or go.norm() < 1e-6:
                continue
            r = _rel(g.float(), go)
            worst = max(worst, (k, r), key=lambda t: t[1])
            assert r < (0.3 if go.numel() == 1 else 0.12), (k, r)
        print("boundary through the TextKV handle: worst parameter-gradient rel L2", worst)
        opt.zero_grad()                                          # a second iteration: DDP's reducer was re-armed
        with torch.amp.autocast("cuda"):
            loss2 = rollout_loss(lambda **kw: ddp(**kw), steps, sels, True)
        scaler.scale(loss2).backward()
        scaler.step(opt)
        scaler.update()
        assert torch.isfinite(loss2).item()
    finally:
        if own_pg:
            dist.destroy_process_group()
