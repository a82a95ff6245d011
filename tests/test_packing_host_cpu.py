"""CPU: the product's host packer (etpnav_b200/packing.py: flatten_gmaps, heading_from_quaternion) and the geometry
code the etp_gmap_pack kernel runs (etpnav_b200/csrc/gmap_pack.cuh, compiled here for the HOST by
tests/host_harness/gmap_pack_host.cpp — test infrastructure, not shipped) against the fixtures the unmodified reference
produced (tests/golden/packing).  Distances / step ids / masks bit-exact; sin / cos of the float32 angles within 1 ulp
(libm sinf vs numpy's float32 sin)."""
import ctypes as C
import os
import subprocess
import types

import numpy as np
import pytest
import torch

from etpnav_b200 import packing
from oracle import packing_port as PK
from tests.test_packing_cpu import cpu_gmap_names, gmap_names, load

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def harness():
    out = os.path.join(HERE, "_build")
    os.makedirs(out, exist_ok=True)
    so = os.path.join(out, "libgmap_pack_host.so")
    src = os.path.join(HERE, "host_harness", "gmap_pack_host.cpp")
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", "-o", so, src], check=True)
    L = C.CDLL(so)
    L.gmap_pack_host.argtypes = [C.c_void_p] * 3 + [C.c_int, C.c_int] + [C.c_void_p] * 5
    return L


def fake_gmaps(gold):
    """GraphMap-shaped objects (dictionaries keyed by viewpoint id) rebuilt from the fixture's plain-data states."""
    gms, cur_vp, cur_pos, cur_ori = [], [], [], []
    for s in gold["states"]:
        nid, gid = s["node_ids"], s["ghost_ids"]
        gm = types.SimpleNamespace(
            node_pos={v: s["node_pos"][k] for k, v in enumerate(nid)},
            ghost_pos={v: None for v in gid},
            ghost_aug_pos={v: s["ghost_pos"][k] for k, v in enumerate(gid)},
            node_stepId={v: int(s["node_step"][k]) for k, v in enumerate(nid)},
            ghost_fronts={v: [nid[f] for f in s["ghost_fronts"][k]] for k, v in enumerate(gid)},
            shortest_dist={a: {b: float(s["dist"][i, j]) for j, b in enumerate(nid)} for i, a in enumerate(nid)},
            shortest_path={a: {b: [0] * int(s["path_len"][i, j]) for j, b in enumerate(nid)} for i, a in enumerate(nid)},
            node_embeds={v: s["node_embeds"][k] for k, v in enumerate(nid)},
            ghost_embeds={v: list(s["ghost_embeds"][k]) for k, v in enumerate(gid)})
        gms.append(gm)
        cur_vp.append(nid[s["cur_node"]])
        cur_pos.append(s["cur_pos"])
        cur_ori.append(s["cur_ori"])
    return gms, cur_vp, cur_pos, cur_ori


def run_host(L, meta, f64, i32b, n_max):
    B = meta.shape[0]
    step = np.empty((B, n_max), dtype=np.int64)
    vis = np.empty((B, n_max), dtype=np.uint8)
    msk = np.empty((B, n_max), dtype=np.uint8)
    pos = np.empty((B, n_max, 7), dtype=np.float32)
    pd = np.empty((B, n_max, n_max), dtype=np.float32)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    meta, f64, i32b = np.ascontiguousarray(meta), np.ascontiguousarray(f64), np.ascontiguousarray(i32b)
    assert L.gmap_pack_host(p(meta), p(f64), p(i32b), B, n_max, p(step), p(vis), p(msk), p(pos), p(pd)) == 0
    return step, vis, msk, pos, pd


@pytest.mark.parametrize("name", cpu_gmap_names())
def test_flatten_and_device_geometry_match_reference(harness, name):
    gold = load(name)
    gms, cur_vp, cur_pos, cur_ori = fake_gmaps(gold)
    meta, f64, i32b, vp_ids, n_max, max_g = packing.flatten_gmaps(gms, cur_vp, cur_pos, cur_ori)
    ref = gold["out"]
    assert vp_ids == ref["gmap_vp_ids"] and n_max == ref["gmap_step_ids"].shape[1]
    assert max_g == max(len(s["ghost_ids"]) for s in gold["states"])
    step, vis, msk, pos, pd = run_host(harness, meta, f64, i32b, n_max)
    assert np.array_equal(step, ref["gmap_step_ids"].numpy())
    assert np.array_equal(vis.astype(bool), ref["gmap_visited_masks"].numpy())
    assert np.array_equal(msk.astype(bool), ref["gmap_masks"].numpy())
    assert np.array_equal(pd, ref["gmap_pair_dists"].numpy()), np.abs(pd - ref["gmap_pair_dists"].numpy()).max()
    rp = ref["gmap_pos_fts"].numpy()
    assert np.array_equal(pos[..., 4:], rp[..., 4:])                      # distances / steps: bit-exact
    assert np.abs(pos[..., :4] - rp[..., :4]).max() <= 1.2e-7             # sin / cos: 1 ulp of float32 at |x| <= 1


def test_heading_matches_oracle_restatement():
    rng = np.random.default_rng(0)
    for _ in range(200):
        q = rng.normal(size=4)
        q /= np.linalg.norm(q)
        a, b = packing.heading_from_quaternion(q), PK.heading_from_quaternion(q)
        assert min(abs(a - b), 2 * np.pi - abs(a - b)) < 1e-12


def test_img_fts_and_vp_index_construction_cpu():
    """The CSR the packers hand to etp_segment_gather, applied densely on the CPU, equals the reference tensors."""
    from etpnav_b200.pretrain import Csr
    captured = []
    orig = packing.segment_gather

    def dense(pool, csr: Csr):
        captured.append(csr)
        out = torch.zeros(csr.num_segments, pool.shape[1])
        for s in range(csr.num_segments):
            for k in range(csr.seg_ptr[s], csr.seg_ptr[s + 1]):
                out[s] += float(csr.weight[k]) * pool[csr.index[k]]
        return out
    packing.segment_gather = dense
    try:
        for name in ("gmap_mid", "edge_gmap"):
            gold = load(name)
            gms, *_ = fake_gmaps(gold)
            n_max = gold["out"]["gmap_step_ids"].shape[1]
            img = packing.pack_gmap_img_fts(gms, n_max, "cpu")
            torch.testing.assert_close(img, gold["out"]["gmap_img_fts"], rtol=1e-6, atol=1e-6)  # x * (1/c) vs x / c
        vp = load("vp_small")
        out = packing.pack_vp_features(vp["obs"], "cpu")
        for k, v in vp["out"].items():
            assert out[k].dtype == v.dtype and torch.equal(out[k], v), k
    finally:
        packing.segment_gather = orig
