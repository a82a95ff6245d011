"""CPU: the packing oracle (oracle/packing_port.py) reproduces what the UNMODIFIED reference packing code produced
(tests/golden/packing, oracle/make_golden_packing.py): ETPTrainer._nav_gmap_variable / _vp_feature_variable and
GraphMap.get_pos_fts.  Bit-exact: the port follows the reference's numpy operation order."""
import glob
import os

import numpy as np
import pytest
import torch

from oracle import packing_port as PK

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "packing")


def load(name):
    return torch.load(os.path.join(GOLD, name + ".pt"), weights_only=False)


def states_of(gold):
    sts = [PK.MapState(s["node_ids"], s["node_pos"], s["node_step"], s["ghost_ids"], s["ghost_pos"], s["ghost_fronts"],
                       s["dist"], s["path_len"]) for s in gold["states"]]
    return sts, gold["states"]


def gmap_names():
    return sorted(os.path.splitext(os.path.basename(p))[0] for p in glob.glob(os.path.join(GOLD, "gmap_*.pt")))


def cpu_gmap_names():
    """gmap_* fixtures (also used by the GPU tests) + the CPU-only edge fixture: ghosts never merged, a map whose ghosts
    have all been explored (no_vp_left), a single-step map."""
    return gmap_names() + ["edge_gmap"]


@pytest.mark.parametrize("name", cpu_gmap_names())
def test_nav_gmap_variable_port_is_bit_exact(name):
    gold = load(name)
    sts, raw = states_of(gold)
    got = PK.nav_gmap_variable(sts, [r["cur_node"] for r in raw], [r["cur_pos"] for r in raw], [r["cur_ori"] for r in raw],
                               [r["node_embeds"] for r in raw], [r["ghost_embeds"] for r in raw])
    ref = gold["out"]
    assert got["gmap_vp_ids"] == ref["gmap_vp_ids"] and got["no_vp_left"] == ref["no_vp_left"]
    for k in ("gmap_step_ids", "gmap_masks", "gmap_visited_masks", "gmap_pair_dists", "gmap_pos_fts", "gmap_img_fts"):
        assert got[k].dtype == ref[k].dtype and got[k].shape == ref[k].shape, k
        assert torch.equal(got[k], ref[k]), (k, (got[k].float() - ref[k].float()).abs().max())


def test_vp_feature_variable_port_is_bit_exact():
    gold = load("vp_small")
    o = gold["obs"]
    got = PK.vp_feature_variable(o["cand_rgb"], o["cand_depth"], o["cand_angle_fts"], o["cand_img_idxes"], o["pano_rgb"],
                                 o["pano_depth"], o["pano_angle_fts"])
    for k, v in gold["out"].items():
        assert got[k].dtype == v.dtype and torch.equal(got[k], v), k


def test_heading_from_quaternion_restatement():
    # yaw rotation about the up axis by theta: heading == theta (habitat convention, nav.py:356 of v0.1.7)
    for th in np.linspace(0.0, 6.2, 17):
        q = [0.0, np.sin(th / 2), 0.0, np.cos(th / 2)]
        assert abs(PK.heading_from_quaternion(q) - th % (2 * np.pi)) < 1e-12
