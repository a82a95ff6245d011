"""Generate tests/golden/packing/*.pt by running the UNMODIFIED reference packing code (oracle/ref_import.py).

TEST INFRASTRUCTURE.  Usage:  python -m oracle.make_golden_packing
Episodes are simulated on the reference's own ``GraphMap`` (vlnce_baselines/models/graph_utils.py:133, imported as is):
random walks that call ``identify_node`` / ``update_graph`` / ``delete_ghost`` the way the rollout does
(ss_trainer_ETP.py:841-869,958), then ``ETPTrainer._nav_gmap_variable`` and ``_vp_feature_variable`` (function bodies
compiled from the reference source, oracle/ref_import.py) produce the tensors.  ``.cuda()`` is made a no-op for the run
(there is no GPU here).  Fixtures store the plain-data map state (oracle/packing_port.py:MapState fields), the
embeddings and the reference's outputs.
"""
import os
import sys
import types

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import packing_port as PK   # noqa: E402
from oracle import ref_import           # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "packing")


def yaw_quat(theta):
    return np.array([0.0, np.sin(theta / 2), 0.0, np.cos(theta / 2)])  # [x, y, z, w], rotation about the up axis


def simulate(gu, rng, g, steps, H, merge_ghost=True, loc_noise=0.5):
    gm = gu.GraphMap(False, loc_noise, merge_ghost, 0)
    pos = rng.normal(0, 2, 3)
    pos[1] = rng.normal(0, 0.1)
    prev = None
    for t in range(steps):
        ori = yaw_quat(rng.uniform(0, 2 * np.pi))
        nc = int(rng.integers(1, 5))
        ang, dis = rng.uniform(0, 2 * np.pi, nc).tolist(), rng.uniform(0.6, 3.0, nc).tolist()
        cur_vp, cand_vp, cand_pos = gm.identify_node(pos, ori, ang, dis)
        gm.update_graph(prev, t + 1, cur_vp, pos, torch.randn(H, generator=g), cand_vp, cand_pos,
                        [torch.randn(H, generator=g) for _ in range(nc)], None)
        last = (cur_vp, pos.copy(), ori)
        if t + 1 < steps:
            gvp = list(gm.ghost_pos.keys())[int(rng.integers(0, len(gm.ghost_pos)))] if gm.ghost_pos else None
            if gvp is None:
                break
            pos = np.array(gm.ghost_mean_pos[gvp], dtype=np.float64) + rng.normal(0, 0.05, 3)
            gm.delete_ghost(gvp)
            gm.ghost_aug_pos.pop(gvp, None)
            prev = cur_vp
    return gm, last


def case_gmap(name, seed, B, max_steps, H=768, edge=False):
    gu = ref_import.load_graph_utils()
    fns = ref_import.load_trainer_packers()
    rng = np.random.default_rng(seed)
    g = torch.Generator().manual_seed(seed)
    gms, cur = [], []
    for i in range(B):
        if edge:
            # 0: ghosts never merged (MODEL.merge_ghost False); 1: every ghost explored away (no_vp_left); 2: a single step
            gm, last = simulate(gu, rng, g, [max_steps, max_steps, 1][i % 3], H, merge_ghost=(i % 3 != 0))
            if i % 3 == 1:
                for gvp in list(gm.ghost_pos.keys()):
                    gm.delete_ghost(gvp)
                    gm.ghost_aug_pos.pop(gvp, None)
        else:
            gm, last = simulate(gu, rng, g, int(rng.integers(1, max_steps + 1)) if i else max_steps, H)
        gms.append(gm)
        cur.append(last)
    fake = types.SimpleNamespace(gmaps=gms, envs=types.SimpleNamespace(num_envs=B))
    out = fns["_nav_gmap_variable"](fake, [c[0] for c in cur], [c[1] for c in cur], [c[2] for c in cur])
    states = []
    for gm, c in zip(gms, cur):
        ms = PK.MapState.from_graph_map(gm)
        states.append(dict(node_ids=ms.node_ids, node_pos=ms.node_pos, node_step=ms.node_step, ghost_ids=ms.ghost_ids,
                           ghost_pos=ms.ghost_pos, ghost_fronts=ms.ghost_fronts, dist=ms.dist, path_len=ms.path_len,
                           cur_node=ms.node_ids.index(c[0]), cur_pos=c[1], cur_ori=c[2],
                           node_embeds=[gm.node_embeds[v] for v in ms.node_ids],
                           ghost_embeds=[(gm.ghost_embeds[v][0], gm.ghost_embeds[v][1]) for v in ms.ghost_ids]))
    os.makedirs(OUT, exist_ok=True)
    torch.save({"name": name, "kind": "gmap", "states": states, "out": out}, os.path.join(OUT, name + ".pt"))
    print(name, "lens", [len(v) for v in out["gmap_vp_ids"]], "pair max", float(out["gmap_pair_dists"].max()))


def case_vp(name, seed, B):
    fns = ref_import.load_trainer_packers()
    g = torch.Generator().manual_seed(seed)
    rng = np.random.default_rng(seed)
    obs = dict(cand_rgb=[], cand_depth=[], cand_angle_fts=[], cand_img_idxes=[], cand_angles=[],
               pano_rgb=torch.randn(B, 12, 512, generator=g), pano_depth=torch.randn(B, 12, 128, generator=g),
               pano_angle_fts=torch.randn(12, 4, generator=g))
    for i in range(B):
        nc = int(rng.integers(1, 6))
        obs["cand_rgb"].append(torch.randn(nc, 512, generator=g))
        obs["cand_depth"].append(torch.randn(nc, 128, generator=g))
        obs["cand_angle_fts"].append(torch.randn(nc, 4, generator=g))
        obs["cand_img_idxes"].append(rng.integers(0, 12, nc))          # duplicates allowed (two waypoints, one sector)
        obs["cand_angles"].append(rng.uniform(0, 6.28, nc).tolist())
    fake = types.SimpleNamespace(envs=types.SimpleNamespace(num_envs=B))
    out = fns["_vp_feature_variable"](fake, obs)
    torch.save({"name": name, "kind": "vp", "obs": obs, "out": out}, os.path.join(OUT, name + ".pt"))
    print(name, "view_lens", out["view_lens"].tolist())


if __name__ == "__main__":
    assert ref_import.available(), "reference not mounted"
    torch.Tensor.cuda = lambda self, *a, **k: self   # no GPU in the authoring container
    case_gmap("gmap_small", 0, 3, 4)
    case_gmap("gmap_mid", 1, 6, 9)
    case_vp("vp_small", 2, 5)
    case_gmap("edge_gmap", 3, 3, 5, edge=True)   # CPU-only fixture (name outside the gmap_* glob of the GPU tests)
