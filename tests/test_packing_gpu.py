"""GPU: caller-side packing (etpnav_b200/packing.py, SURVEY.md §8f N3) through the C ABI against the fixtures produced
by the UNMODIFIED reference packing code (tests/golden/packing): pack_gmap vs ETPTrainer._nav_gmap_variable,
pack_vp_features vs _vp_feature_variable.  Integer / bool tensors and all distances bit-exact; sin / cos within 1 ulp;
image features to fp32 rounding of x * (1/count) vs x / count."""
import numpy as np
import pytest
import torch

from tests.test_packing_cpu import gmap_names, load
from tests.test_packing_host_cpu import fake_gmaps

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(120)]


@pytest.mark.parametrize("name", gmap_names())
def test_pack_gmap_matches_reference(name):
    from etpnav_b200 import packing
    gold = load(name)
    gms, cur_vp, cur_pos, cur_ori = fake_gmaps(gold)
    for gm in gms:   # the maps hold device tensors in the trainer
        gm.node_embeds = {k: v.cuda().requires_grad_(True) for k, v in gm.node_embeds.items()}
        gm.ghost_embeds = {k: [v[0].cuda(), v[1]] for k, v in gm.ghost_embeds.items()}
    out = packing.pack_gmap(gms, cur_vp, cur_pos, cur_ori, device="cuda")
    torch.cuda.synchronize()
    ref = gold["out"]
    assert out["gmap_vp_ids"] == ref["gmap_vp_ids"] and out["no_vp_left"] == ref["no_vp_left"]
    for k in ("gmap_step_ids", "gmap_masks", "gmap_visited_masks", "gmap_pair_dists"):
        assert out[k].dtype == ref[k].dtype and torch.equal(out[k].cpu(), ref[k]), k
    pos, rp = out["gmap_pos_fts"].cpu(), ref["gmap_pos_fts"]
    assert torch.equal(pos[..., 4:], rp[..., 4:])
    assert (pos[..., :4] - rp[..., :4]).abs().max().item() <= 2.4e-7
    torch.testing.assert_close(out["gmap_img_fts"].cpu(), ref["gmap_img_fts"], rtol=1e-6, atol=1e-6)
    # inference path: no tensor requires grad -> the per-node tensors are read in place through a pointer table
    with torch.no_grad():
        img_ng = packing.pack_gmap_img_fts(gms, ref["gmap_img_fts"].shape[1], "cuda")
    assert torch.equal(img_ng, out["gmap_img_fts"].detach())
    # the gather is differentiable: the gradient of a node row lands on that node's embedding
    out["gmap_img_fts"].sum().backward()
    first = next(iter(gms[0].node_embeds.values()))
    assert torch.equal(first.grad.cpu(), torch.ones(768))


def test_pack_vp_features_matches_reference():
    from etpnav_b200 import packing
    gold = load("vp_small")
    o = gold["obs"]
    obs = {k: ([t.cuda() if torch.is_tensor(t) else t for t in v] if isinstance(v, list) else
               (v.cuda() if torch.is_tensor(v) else v)) for k, v in o.items()}
    out = packing.pack_vp_features(obs, device="cuda")
    torch.cuda.synchronize()
    for k, v in gold["out"].items():
        assert out[k].dtype == v.dtype and torch.equal(out[k].cpu(), v), k


def test_pack_gmap_large_random_maps_properties():
    """Maps far larger than the fixtures (up to 120 nodes, B = 64): symmetry, zero diagonal / [stop] row, zero padding,
    agreement with the CPU oracle port on a sample of environments."""
    import types
    from etpnav_b200 import packing
    from oracle import packing_port as PK
    rng = np.random.default_rng(5)
    gms, cur_vp, cur_pos, cur_ori = [], [], [], []
    for e in range(64):
        n, g = int(rng.integers(2, 30)), int(rng.integers(0, 90))
        nid, gid = [str(k) for k in range(n)], [f"g{k}" for k in range(g)]
        P = rng.normal(0, 5, (n, 3))
        D = np.linalg.norm(P[:, None] - P[None], axis=-1)
        gm = types.SimpleNamespace(
            node_pos={v: P[k] for k, v in enumerate(nid)}, ghost_pos={v: None for v in gid},
            ghost_aug_pos={v: rng.normal(0, 5, 3) for v in gid}, node_stepId={v: k + 1 for k, v in enumerate(nid)},
            ghost_fronts={v: [nid[int(f)] for f in rng.integers(0, n, int(rng.integers(1, 4)))] for v in gid},
            shortest_dist={a: {b: float(D[i, j]) for j, b in enumerate(nid)} for i, a in enumerate(nid)},
            shortest_path={a: {b: [0] * (1 + abs(i - j)) for j, b in enumerate(nid)} for i, a in enumerate(nid)})
        gms.append(gm)
        cur_vp.append(nid[int(rng.integers(0, n))])
        cur_pos.append(rng.normal(0, 5, 3))
        th = rng.uniform(0, 6.28)
        cur_ori.append(np.array([0.0, np.sin(th / 2), 0.0, np.cos(th / 2)]))
    meta, f64, i32b, vp_ids, n_max, max_g = packing.flatten_gmaps(gms, cur_vp, cur_pos, cur_ori)
    out = packing.pack_gmap_geometry(meta, f64, i32b, n_max, max_g, "cuda")
    torch.cuda.synchronize()
    pd, msk = out["gmap_pair_dists"].cpu(), out["gmap_masks"].cpu()
    assert torch.equal(pd, pd.transpose(1, 2)) and pd.diagonal(dim1=1, dim2=2).abs().max() == 0
    assert pd[:, 0].abs().max() == 0 and (pd * ~(msk[:, :, None] & msk[:, None, :])).abs().max() == 0
    assert torch.equal(msk.sum(1), torch.tensor([len(v) for v in vp_ids]))
    for e in (0, 17, 63):
        ms = PK.MapState.from_graph_map(gms[e])
        L = len(vp_ids[e])
        assert np.array_equal(pd[e, :L, :L].numpy(), PK.pair_dists(ms))
        want = PK.get_pos_fts(ms, ms.node_ids.index(cur_vp[e]), cur_pos[e], cur_ori[e])
        got = out["gmap_pos_fts"][e, :L].cpu().numpy()
        assert np.array_equal(got[:, 4:], want[:, 4:]) and np.abs(got[:, :4] - want[:, :4]).max() <= 2.4e-7


@pytest.mark.parametrize("name", gmap_names())
def test_stateful_packer_matches_reference_fixtures(name):
    """GmapPacker (incremental mirror, one H2D, two launches) on the reference's fixtures: same gate as pack_gmap."""
    from etpnav_b200 import packing
    gold = load(name)
    gms, cur_vp, cur_pos, cur_ori = fake_gmaps(gold)
    for gm in gms:
        gm.node_embeds = {k: v.cuda() for k, v in gm.node_embeds.items()}
        gm.ghost_embeds = {k: [v[0].cuda(), v[1]] for k, v in gm.ghost_embeds.items()}
    pk = packing.GmapPacker("cuda")
    ref = gold["out"]
    for _ in range(2):            # second call: nothing changed, everything comes from the mirror
        out = pk.pack(gms, cur_vp, cur_pos, cur_ori)
        torch.cuda.synchronize()
        assert out["gmap_vp_ids"] == ref["gmap_vp_ids"] and out["no_vp_left"] == ref["no_vp_left"]
        for k in ("gmap_step_ids", "gmap_masks", "gmap_visited_masks", "gmap_pair_dists"):
            assert out[k].dtype == ref[k].dtype and torch.equal(out[k].cpu(), ref[k]), k
        pos, rp = out["gmap_pos_fts"].cpu(), ref["gmap_pos_fts"]
        assert torch.equal(pos[..., 4:], rp[..., 4:])
        assert (pos[..., :4] - rp[..., :4]).abs().max().item() <= 2.4e-7
        torch.testing.assert_close(out["gmap_img_fts"].cpu(), ref["gmap_img_fts"], rtol=1e-6, atol=1e-6)


def test_stateful_packer_follows_evolving_maps_bit_for_bit():
    """Evolving maps (tests/gmap_sim.py): at every step the stateful packer's six tensors equal the stateless
    pack_gmap's; an embedding that needs a gradient sends the image features through the differentiable gather."""
    from etpnav_b200 import packing
    from tests.gmap_sim import SimGraphMap
    rng = np.random.default_rng(3)
    gms = [SimGraphMap(40 + e, device="cuda").step() for e in range(8)]
    pk = packing.GmapPacker("cuda")
    keys = ("gmap_step_ids", "gmap_visited_masks", "gmap_masks", "gmap_pos_fts", "gmap_pair_dists", "gmap_img_fts")
    for t in range(14):
        cur_vp, cur_pos, cur_ori = (list(x) for x in zip(*[gm.pose() for gm in gms]))
        with torch.no_grad():
            out = pk.pack(gms, cur_vp, cur_pos, cur_ori)
            ref = packing.pack_gmap(gms, cur_vp, cur_pos, cur_ori, "cuda")
        for k in keys:
            assert torch.equal(out[k], ref[k]), (t, k)
        assert out["gmap_vp_ids"] == ref["gmap_vp_ids"] and out["no_vp_left"] == ref["no_vp_left"]
        for gm in gms:
            if rng.random() < 0.8:
                gm.step()
        if t == 6:
            gms.pop(3)
        if t == 9:
            gms[0] = SimGraphMap(777, device="cuda").step()
    gm = gms[1]
    v = next(iter(gm.node_embeds))
    gm.step()
    new = list(gm.node_embeds)[-1]
    gm.node_embeds[new] = gm.node_embeds[new].clone().requires_grad_(True)
    cur_vp, cur_pos, cur_ori = (list(x) for x in zip(*[g.pose() for g in gms]))
    out = pk.pack(gms, cur_vp, cur_pos, cur_ori)
    out["gmap_img_fts"].sum().backward()
    assert torch.equal(gm.node_embeds[new].grad.cpu(), torch.ones(768))
