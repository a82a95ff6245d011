"""CPU restatement of the trainer's caller-side packing (SURVEY.md §8f N3) — TEST INFRASTRUCTURE, not product code.

numpy / torch-CPU restatement of (paths relative to /root/reference/vlnce_baselines)
  ETPTrainer._vp_feature_variable   ss_trainer_ETP.py:308-342
  ETPTrainer._nav_gmap_variable     ss_trainer_ETP.py:344-417
  GraphMap.get_pos_fts / front_to_ghost_dist / get_node_embeds   models/graph_utils.py:258-322
  calculate_vp_rel_pos_fts / get_angle_fts / heading_from_quaternion   models/graph_utils.py:21-58
operating on a plain-data view of a GraphMap (``MapState`` below).  ``heading_from_quaternion`` depends on
habitat-lab v0.1.7 (``habitat.utils.geometry_utils.quaternion_from_coeff / quaternion_rotate_vector``,
``habitat.tasks.utils.cartesian_to_polar``; the reference pins habitat-lab 0.1.7, README "Installation") and
numpy-quaternion, both absent from /root/reference: their published algorithm (Hamilton product q v q^-1, coefficients
ordered [x, y, z, w]; polar angle = arctan2(y, x)) is restated in ``heading_from_quaternion``.
Pinned by ``oracle/make_golden_packing.py``, which runs the reference's own GraphMap and the two trainer methods (the
function bodies are executed from the reference source, unmodified) -> ``tests/golden/packing/*.pt``.
"""
import numpy as np
import torch

MAX_DIST, MAX_STEP = 30, 10  # graph_utils.py:9-10


def quat_mul(a, b):
    # Hamilton product, (w, x, y, z)
    aw, ax, ay, az = a
    bw, bx, by, bz = b
    return np.array([aw * bw - ax * bx - ay * by - az * bz,
                     aw * bx + ax * bw + ay * bz - az * by,
                     aw * by - ax * bz + ay * bw + az * bx,
                     aw * bz + ax * by - ay * bx + az * bw])


def quat_inverse(q):
    return np.array([q[0], -q[1], -q[2], -q[3]]) / float(np.dot(q, q))


def quaternion_rotate_vector(q, v):
    # habitat-lab v0.1.7 habitat/utils/geometry_utils.py: (quat * vq * quat.inverse()).imag
    vq = np.array([0.0, v[0], v[1], v[2]])
    return quat_mul(quat_mul(q, vq), quat_inverse(q))[1:]


def heading_from_quaternion(coeffs):
    # graph_utils.py:53-58; coeffs = [x, y, z, w] (quaternion_from_coeff)
    q = np.array([coeffs[3], coeffs[0], coeffs[1], coeffs[2]], dtype=np.float64)
    hv = quaternion_rotate_vector(quat_inverse(q), np.array([0.0, 0.0, -1.0]))
    phi = np.arctan2(hv[0], -hv[2])  # cartesian_to_polar(-hv[2], hv[0])[1]
    return phi % (2 * np.pi)


def position_distance(a, b):
    # graph_utils.py:13-19
    dx, dy, dz = b[0] - a[0], b[1] - a[1], b[2] - a[2]
    return np.sqrt(dx ** 2 + dy ** 2 + dz ** 2)


class MapState:
    """Plain-data view of one GraphMap at one step (what the host packer flattens): node / ghost ids in dictionary
    order, positions, step ids, fronts (node indices), all-pairs shortest distance and path length between nodes."""

    def __init__(self, node_ids, node_pos, node_step, ghost_ids, ghost_pos, ghost_fronts, dist, path_len):
        self.node_ids, self.ghost_ids = list(node_ids), list(ghost_ids)
        self.node_pos = np.asarray(node_pos, dtype=np.float64).reshape(-1, 3)
        self.ghost_pos = np.asarray(ghost_pos, dtype=np.float64).reshape(-1, 3)
        self.node_step = np.asarray(node_step, dtype=np.int64)
        self.ghost_fronts = [list(f) for f in ghost_fronts]
        self.dist = np.asarray(dist, dtype=np.float64).reshape(len(self.node_ids), len(self.node_ids))
        self.path_len = np.asarray(path_len, dtype=np.int64).reshape(len(self.node_ids), len(self.node_ids))

    @classmethod
    def from_graph_map(cls, gmap):
        """From a reference ``GraphMap`` (or anything with its attributes)."""
        nid, gid = list(gmap.node_pos.keys()), list(gmap.ghost_pos.keys())
        ix = {vp: i for i, vp in enumerate(nid)}
        n = len(nid)
        dist, plen = np.zeros((n, n)), np.zeros((n, n), dtype=np.int64)
        for a in nid:
            for b in nid:
                dist[ix[a], ix[b]] = gmap.shortest_dist[a][b]
                plen[ix[a], ix[b]] = len(gmap.shortest_path[a][b])
        return cls(nid, [gmap.node_pos[v] for v in nid], [gmap.node_stepId[v] for v in nid], gid,
                   [gmap.ghost_aug_pos[v] for v in gid], [[ix[f] for f in gmap.ghost_fronts[v]] for v in gid], dist, plen)

    def front_to_ghost_dist(self, g):
        # graph_utils.py:258-270
        best, bf = 10000, None
        for f in self.ghost_fronts[g]:
            d = position_distance(self.node_pos[f], self.ghost_pos[g])
            if d < best:
                best, bf = d, f
        return best, bf


def rel_pos(a, b, base_heading):
    # calculate_vp_rel_pos_fts (graph_utils.py:21-45) with base_elevation = 0, to_clock = True
    dx, dy, dz = b[0] - a[0], b[1] - a[1], b[2] - a[2]
    xz = max(np.sqrt(dx ** 2 + dz ** 2), 1e-8)
    xyz = max(np.sqrt(dx ** 2 + dy ** 2 + dz ** 2), 1e-8)
    heading = np.arcsin(-dx / xz)
    if b[2] > a[2]:
        heading = np.pi - heading
    heading -= base_heading
    heading = 2 * np.pi - heading
    return heading, np.arcsin(dz / xyz), xyz


def get_pos_fts(ms, cur_node, cur_pos, cur_ori):
    """GraphMap.get_pos_fts (graph_utils.py:278-322) for gmap_vp_ids = [None] + nodes + ghosts -> float32 [len, 7]."""
    cur_pos = np.asarray(cur_pos, dtype=np.float64)
    base = heading_from_quaternion(cur_ori)
    ang, dis = [[0, 0]], [[0, 0, 0]]
    for k in range(len(ms.node_ids)):
        h, e, d = rel_pos(cur_pos, ms.node_pos[k], base)
        ang.append([h, e])
        dis.append([d / MAX_DIST, ms.dist[cur_node, k] / MAX_DIST, ms.path_len[cur_node, k] / MAX_STEP])
    for g in range(len(ms.ghost_ids)):
        h, e, d = rel_pos(cur_pos, ms.ghost_pos[g], base)
        ang.append([h, e])
        fd, f = ms.front_to_ghost_dist(g)
        dis.append([d / MAX_DIST, (ms.dist[cur_node, f] + fd) / MAX_DIST, (ms.path_len[cur_node, f] + 1) / MAX_STEP])
    ang = np.array(ang).astype(np.float32)
    dis = np.array(dis).astype(np.float32)
    fts = np.vstack([np.sin(ang[:, 0]), np.cos(ang[:, 0]), np.sin(ang[:, 1]), np.cos(ang[:, 1])]).transpose().astype(np.float32)
    return np.concatenate([fts, dis], 1)


def pair_dists(ms):
    """ss_trainer_ETP.py:371-387 -> float32 [len, len]."""
    n, g = len(ms.node_ids), len(ms.ghost_ids)
    L = 1 + n + g
    out = np.zeros((L, L), dtype=np.float32)
    fr = [ms.front_to_ghost_dist(k) for k in range(g)]
    for j in range(1, L):
        for k in range(j + 1, L):
            gj, gk = j > n, k > n
            if not gj and not gk:
                d = ms.dist[j - 1, k - 1]
            elif not gj and gk:
                fd2, f2 = fr[k - 1 - n]
                d = ms.dist[j - 1, f2] + fd2
            else:
                fd1, f1 = fr[j - 1 - n]
                fd2, f2 = fr[k - 1 - n]
                d = fd1 + ms.dist[f1, f2] + fd2
            out[j, k] = out[k, j] = d / MAX_DIST
    return out


def nav_gmap_variable(states, cur_nodes, cur_pos, cur_ori, node_embeds, ghost_embeds):
    """_nav_gmap_variable (ss_trainer_ETP.py:344-417) on MapStates.  node_embeds[i]: list of [H] tensors in node order;
    ghost_embeds[i]: list of (sum tensor, count) in ghost order (get_node_embeds, graph_utils.py:272-276)."""
    B = len(states)
    lens = [1 + len(s.node_ids) + len(s.ghost_ids) for s in states]
    N = max(lens)
    H = node_embeds[0][0].shape[0]
    step_ids = torch.zeros(B, N, dtype=torch.long)
    visited = torch.zeros(B, N, dtype=torch.bool)
    img = torch.zeros(B, N, H)
    pos = torch.zeros(B, N, 7)
    pd = torch.zeros(B, N, N)
    vp_ids = []
    for i, s in enumerate(states):
        n = len(s.node_ids)
        vp_ids.append([None] + s.node_ids + s.ghost_ids)
        step_ids[i, 1:1 + n] = torch.from_numpy(s.node_step)
        visited[i, 1:1 + n] = True
        rows = list(node_embeds[i]) + [e / c for e, c in ghost_embeds[i]]
        img[i, 1:lens[i]] = torch.stack(rows, 0)
        pos[i, :lens[i]] = torch.from_numpy(get_pos_fts(s, cur_nodes[i], cur_pos[i], cur_ori[i]))
        pd[i, :lens[i], :lens[i]] = torch.from_numpy(pair_dists(s))
    masks = torch.arange(N)[None] < torch.tensor(lens)[:, None]
    return dict(gmap_vp_ids=vp_ids, gmap_step_ids=step_ids, gmap_img_fts=img, gmap_pos_fts=pos, gmap_masks=masks,
                gmap_visited_masks=visited, gmap_pair_dists=pd, no_vp_left=[len(s.ghost_ids) == 0 for s in states])


def vp_feature_variable(cand_rgb, cand_depth, cand_angle_fts, cand_img_idxes, pano_rgb, pano_depth, pano_angle_fts):
    """_vp_feature_variable (ss_trainer_ETP.py:308-342): candidate views first, then the non-candidate panorama views."""
    B = len(cand_rgb)
    rgb, dep, loc, nav, lens = [], [], [], [], []
    for i in range(B):
        is_cand = np.zeros(12, dtype=bool)
        is_cand[cand_img_idxes[i]] = True
        keep = torch.from_numpy(~is_cand)
        rgb.append(torch.cat([cand_rgb[i], pano_rgb[i][keep]], 0))
        dep.append(torch.cat([cand_depth[i], pano_depth[i][keep]], 0))
        loc.append(torch.cat([cand_angle_fts[i], pano_angle_fts[keep]], 0))
        nav.append([1] * len(cand_rgb[i]) + [0] * int(12 - is_cand.sum()))
        lens.append(len(nav[-1]))
    V = max(lens)

    def pad(ts):
        out = torch.zeros(B, V, ts[0].shape[1])
        for i, t in enumerate(ts):
            out[i, :len(t)] = t
        return out
    nt = torch.zeros(B, V, dtype=torch.long)
    for i, x in enumerate(nav):
        nt[i, :len(x)] = torch.tensor(x)
    return dict(rgb_fts=pad(rgb), dep_fts=pad(dep), loc_fts=pad(loc), nav_types=nt, view_lens=torch.tensor(lens))
