"""Training-rollout benchmark of the episode-level text K|V handle (DESIGN.md §5a).

    python profiles/rollout_bench.py [--repeats 7] [--warmup 3] [--out profiles/r03_rollout_textkv.json]

Workload: what the reference trainer runs per iteration (ss_trainer_ETP.py:801-892, :504) at the c3 shapes (B 64, 12 views,
200 tokens, 9 language / 2 panorama / 6 cross-modal layers), train() with dropout on: forward_txt once, then for T = 15
steps forward_panorama and forward_navigation on the surviving episodes (the map grows to N = 80 nodes; episodes finish
from step 5 on, 64 -> 44), the CE of every step summed into one loss, ONE backward, torch AdamW.  The un-cached rollout
indexes txt_embeds[not_done_index] at each step; the handle rollout indexes encode_text_kv(txt_embeds) instead.

Both rollouts run in this process, alternating, `--repeats` times each after `--warmup` rounds; each is timed with a
device synchronise on both ends, and torch.cuda.max_memory_allocated is reset before it.  A separate torch.profiler run of
one rollout of each kind gives the kernel totals: GEMM time of each kind (their difference is what the handle saves on the
text side, net of its own once-per-rollout GEMMs) and the accumulation kernel.  Needs a CUDA device: there is no CPU path.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.dont_write_bytecode = True

import torch  # noqa: E402

B0, V, L, X, NL, T, N_END = 64, 12, 200, 6, 9, 15, 80


def _alive(t):
    return B0 - 2 * max(0, t - 4)


def _card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), "r03_rollout_textkv.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("rollout_bench.py needs a CUDA device")
    from etpnav_b200.config import PlannerConfig
    from etpnav_b200.planner import B200Planner
    from etpnav_b200.synth import make_inputs, make_weights

    torch.manual_seed(0)
    cfg = PlannerConfig(num_l_layers=NL, num_x_layers=X)
    m = B200Planner(cfg, device="cuda")
    m.load_state_dict(make_weights(cfg, seed=3), strict=True)
    m.train()
    opt = torch.optim.AdamW(m.parameters(), lr=1e-5)
    finish = torch.randperm(B0, generator=torch.Generator().manual_seed(5)).tolist()  # order in which episodes end
    steps = []
    for t in range(T):
        n = round(8 + (N_END - 8) * t / (T - 1))
        inp = make_inputs(cfg, B0, V, n, L, seed=100 + t, ragged=True)
        d = {k: (v.cuda() if isinstance(v, torch.Tensor) else v) for k, v in inp.items()}
        d["sel"] = sorted(finish[B0 - _alive(t):])                                         # not_done_index (a list)
        steps.append(d)
    d0 = steps[0]

    def rollout(handle):
        txt = m.forward_txt(d0["txt_ids"], d0["txt_masks"])
        src = m.encode_text_kv(txt) if handle else txt
        loss = 0.0
        for d in steps:
            sel = d["sel"]
            pano, pm = m.forward_panorama(d["rgb_fts"][sel], d["dep_fts"][sel], d["loc_fts"][sel], d["nav_types"][sel],
                                          d["view_lens"][sel])
            w = pm.unsqueeze(-1).to(pano.dtype)
            img = d["gmap_img_fts"][sel].clone()
            img[:, 1] = img[:, 1] + (pano * w).sum(1) / w.sum(1)
            out = m.forward_navigation(src[sel], d0["txt_masks"][sel], None, d["gmap_step_ids"][sel], img,
                                       d["gmap_pos_fts"][sel], d["gmap_masks"][sel], d["gmap_visited_masks"][sel],
                                       d["gmap_pair_dists"][sel])
            loss = loss + torch.nn.functional.cross_entropy(out["global_logits"], d["labels"][sel], reduction="sum")
        loss.backward()
        opt.step()
        opt.zero_grad(set_to_none=True)
        return loss

    def timed(handle):
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        t0 = time.perf_counter()
        loss = rollout(handle)
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3, torch.cuda.max_memory_allocated() - base, loss.item()

    res = {"uncached": {"ms": [], "peak_bytes": [], "loss": []}, "handle": {"ms": [], "peak_bytes": [], "loss": []}}
    for r in range(a.warmup + a.repeats):
        for kind in (("uncached", "handle") if r % 2 == 0 else ("handle", "uncached")):
            ms, peak, loss = timed(kind == "handle")
            if r >= a.warmup:
                res[kind]["ms"].append(round(ms, 3))
                res[kind]["peak_bytes"].append(peak)
                res[kind]["loss"].append(loss)

    # kernel totals from a profiler run of its own
    from torch.profiler import ProfilerActivity, profile
    kernels = {}
    for kind in ("uncached", "handle"):
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            rollout(kind == "handle")
            torch.cuda.synchronize()
        tot = {}
        for e in prof.key_averages():
            if e.device_time_total > 0:
                tot[e.key] = (tot.get(e.key, (0.0, 0))[0] + e.device_time_total / 1e3, e.count)
        gemm = sum(v[0] for k, v in tot.items() if "gemm" in k.lower())
        acc = sum(v[0] for k, v in tot.items() if "kv_grad_accumulate" in k)
        top = sorted(tot.items(), key=lambda kv: -kv[1][0])[:12]
        kernels[kind] = {"gemm_ms": round(gemm, 3), "kv_grad_accumulate_ms": round(acc, 3),
                         "kv_grad_accumulate_launches": sum(v[1] for k, v in tot.items() if "kv_grad_accumulate" in k),
                         "all_kernels_ms": round(sum(v[0] for v in tot.values()), 3),
                         "top": [{"kernel": k[:120], "ms": round(v[0], 3), "launches": v[1]} for k, v in top]}

    def summary(k):
        ms = res[k]["ms"]
        return {"ms_per_rollout_median": round(statistics.median(ms), 3), "ms_per_rollout": ms,
                "max_memory_allocated_gb_median": round(statistics.median(res[k]["peak_bytes"]) / 1e9, 3),
                "loss": res[k]["loss"]}

    out = {
        "workload": {"batch": B0, "views": V, "tokens": L, "l_layers": NL, "x_layers": X, "steps": T, "nodes_end": N_END,
                     "alive_per_step": [_alive(t) for t in range(T)], "dropout": True, "optimizer": "torch.optim.AdamW"},
        "card": _card(),
        "repeats": a.repeats, "warmup": a.warmup,
        "uncached": summary("uncached"), "handle": summary("handle"),
        "profiler": kernels,
        "gemm_ms_saved_per_rollout": round(kernels["uncached"]["gemm_ms"] - kernels["handle"]["gemm_ms"], 3),
        "note": "peak = max_memory_allocated during the rollout above what was allocated before it; profiler totals come "
                "from one separate traced rollout of each kind",
    }
    out["handle_vs_uncached_time"] = round(out["handle"]["ms_per_rollout_median"] / out["uncached"]["ms_per_rollout_median"], 4)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: out[k] for k in ("card", "handle_vs_uncached_time", "gemm_ms_saved_per_rollout")}
                     | {"uncached_ms": out["uncached"]["ms_per_rollout_median"], "handle_ms": out["handle"]["ms_per_rollout_median"],
                        "uncached_peak_gb": out["uncached"]["max_memory_allocated_gb_median"],
                        "handle_peak_gb": out["handle"]["max_memory_allocated_gb_median"]}))


if __name__ == "__main__":
    main()
