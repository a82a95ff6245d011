#!/usr/bin/env python
"""Planner-step benchmark (contract: one JSON line on rank 0).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--mode train|fwd] [--dump-outputs DIR]

Metric (BASELINE.json): planner steps/s at B=64 episodes per GPU, 12 views, 80-node graph, 200-token
instruction, 6 cross-modal layers (BASELINE.json configs[2]; the reference checkpoints use 4 — pass
``--x-layers 4``).  One *planner step* = forward_panorama + forward_navigation (+ backward of both and one
AdamW update in ``train`` mode) on a batch of B episodes (SURVEY.md §8d).  Synthetic seeded tensors
(etpnav_b200/synth.py), random-init weights of the reference architecture.

* ``value``  — steps/s with the step's inputs already resident in HBM (CUDA-event time over exactly K
  steps, max over ranks, barrier + synchronize on both sides).
* ``e2e``    — the same metric through the public module API with HOST inputs: pinned-host -> device copies
  of every input tensor and a device -> host read of the node logits inside the timed region.
* ``roofline`` — tcgen05 GEMM kernel: algorithmic FLOPs of its launches / their CUDA-event time (measured
  in a separate profiled pass of the same step) against the measured bf16 peak of MEASURED_PEAKS.json.
* ``cpu_baseline`` — the oracle port of the reference (oracle/planner_port.py, fp32, all host cores) on a
  bounded sample of the same workload.  ``--impl reference`` runs ONLY that CPU arm.
Data-parallel (N > 1): every rank runs its own batch of B episodes (weak scaling); in ``train`` mode the
flat gradient buffer of the step's parameters is all-reduced once over NCCL before AdamW.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree it runs from (it may be read-only)

from etpnav_b200.config import PlannerConfig            # noqa: E402
from etpnav_b200.synth import make_inputs, make_weights, step_flops  # noqa: E402



# BASELINE.json configurations that are bench lines (the others are parity-test cases): per-GPU shapes
PRESETS = {
    # configs[2] — the metric's own configuration (SIX cross-modal layers as BASELINE.json words it)
    "c3": dict(batch=64, views=12, nodes=80, tokens=200, x_layers=6, text_law=None, xlmr=False),
    # configs[3] — 8 x 64 episodes, R2R-CE instruction-length law (IL.max_text_len 80, run_r2r/iter_train.yaml:42), 4 layers
    "c4": dict(batch=64, views=12, nodes=80, tokens=80, x_layers=4, text_law="r2r", xlmr=False),
    # configs[4] — RxR-CE shape: XLM-R (eps 1e-5, 514 positions), 512-token instruction, 120-node graph, 8 x 32 episodes
    "c5": dict(batch=32, views=12, nodes=120, tokens=512, x_layers=4, text_law=None, xlmr=True),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--mode", default=None, choices=["train", "fwd"])
    ap.add_argument("--config", default="c3", choices=sorted(PRESETS),
                    help="BASELINE.json configuration: c3 (default, the metric's own), c4 (R2R-CE lengths), c5 (RxR-CE / XLM-R shape)")
    ap.add_argument("--batch", type=int, default=None)
    ap.add_argument("--views", type=int, default=None)
    ap.add_argument("--nodes", type=int, default=None)
    ap.add_argument("--tokens", type=int, default=None)
    ap.add_argument("--x-layers", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dropout", default="on", choices=["on", "off"],
                    help="train mode: the reference's train() dropout (0.1 hidden / attention / head) on (default) or off")
    ap.add_argument("--gpu-eager", action="store_true", help="(default on at N=1; kept for old command lines)")
    ap.add_argument("--no-gpu-eager", action="store_true",
                    help="skip the eager-PyTorch-on-this-GPU legs (fp32 and bf16 autocast): the 'reference GPU eager' figure "
                         "the north_star's >=10x target is stated against")
    ap.add_argument("--no-soak", action="store_true", help="skip the >= 3 s sustained run (clocks / power under a long region)")
    ap.add_argument("--no-dp-check", action="store_true", help="N > 1: skip the data-parallel gradient self-check step")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "high"],
                    help="fwd mode: 'high' = the fp32-class inference mode (split-bf16 x3 GEMMs + fp32 attention)")
    ap.add_argument("--text-kv", action="store_true",
                    help="fwd mode: the instruction's key|value projections are computed once per episode "
                         "(B200Planner.encode_text_kv, outside the timed step) and reused by every step, as in an eval rollout")
    ap.add_argument("--grad-comm", default="peer", choices=["fp32", "bf16", "peer"],
                    help="N > 1: peer (default) = reduce-scatter + AdamW + parameter all-gather fused in one kernel per bucket "
                         "over NVLink peer memory (falls back to fp32 when CUDA IPC / peer access is unavailable) | fp32 = NCCL "
                         "all-reduce of the gradient buckets + replicated AdamW (DDP's arithmetic) | bf16 = the same in bf16")
    ap.add_argument("--peer-ctas", type=int, default=128, help="N > 1, --grad-comm peer: grid of the fused update kernel")
    ap.add_argument("--comm-sms", type=int, default=0,
                    help="N > 1: SMs the persistent grids leave to the collective (etp_set_sm_reserve)")
    ap.add_argument("--nccl-max-ctas", type=int, default=0, help="N > 1: NCCL_MAX_CTAS for this run (0 = NCCL's default)")
    ap.add_argument("--kernel-report", default=None, help="write the per-kernel CUDA-event table of the profiled pass here")
    ap.add_argument("--text-law", default=None, choices=["r2r"],
                    help="ragged instruction lengths: 'r2r' = normal(32, 12) clipped to [8, 80] BERT tokens (BASELINE.json "
                         "configs[3]; etpnav_b200/synth.py:r2r_text_lengths), padded to --tokens")
    ap.add_argument("--workload", default="planner", choices=["planner", "pretrain", "packing"],
                    help="planner (default, BASELINE.json's metric) | pretrain (SURVEY.md 8f N2: one pre-training iteration "
                         "of the twin, mlm and sap alternating) | packing (8f N3: the per-step map / view packing)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="planner workload: after the timed steps write what the last timed step computed as DIR/<name>.npy "
                         "(float32; the inputs are seeded, so two builds can be compared output for output)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.workload != "planner" or a.impl != "b200"):
        ap.error("--dump-outputs covers the planner workload of the b200 arm")
    pre = PRESETS[a.config]
    for k in ("batch", "views", "nodes", "tokens", "x_layers", "text_law"):
        if getattr(a, k) is None:
            setattr(a, k, pre[k])
    a.xlmr = pre["xlmr"]
    return a


def metric_name(a):
    return f"planner steps/sec (B={a.batch},{a.views}v,{a.nodes}n,{a.tokens}t)"


def workload_cfg(a):
    # text-side tensors are not part of the per-step path: keep the vocab small so set-up is fast
    kw = dict(vocab_size=2048, num_l_layers=0, num_x_layers=a.x_layers)
    if a.xlmr:   # bert_config/xlm-roberta-base/config.json:13 + vlnbert_init.py:32-39
        kw.update(max_position_embeddings=514, layer_norm_eps=1e-5)
    cfg = PlannerConfig(**kw)
    if a.dropout == "off":
        cfg.hidden_dropout_prob = cfg.attention_probs_dropout_prob = cfg.pred_head_dropout_prob = 0.0
    return cfg


def config_dict(a, mode, world):
    """The ``config`` object of the JSON line — built by ONE function for both arms so they compare equal."""
    return {"workload": workload_name(a, mode), "name": a.config, "mode": mode, "global_batch": a.batch * max(1, world),
            "parallelism": f"dp{max(1, world)}", "x_layers": a.x_layers, "dropout": a.dropout if mode == "train" else "n/a",
            "grad_comm": (a.grad_comm if (world > 1 and mode == "train") else "n/a"),
            "l2": "no flush: the per-step working set (activation record + weights, > 1 GB in train mode) exceeds the 126 MB L2"}


def torch_dropout_hook(cfg):
    """drop(x, kind, site) for the oracle port in the baseline legs: torch's own nn.Dropout arithmetic at the
    reference's dropout sites (train mode), or None when every probability is 0."""
    import torch.nn.functional as F
    ps = {"hidden": cfg.hidden_dropout_prob, "attn": cfg.attention_probs_dropout_prob, "head": cfg.pred_head_dropout_prob}
    if max(ps.values()) <= 0:
        return None
    return lambda x, kind, site: F.dropout(x, ps[kind], True)


def workload_name(a, mode):
    what = ("fwd+bwd+AdamW, train() dropout " + a.dropout) if mode == "train" else (
        "fwd (episode-level text K|V cache)" if getattr(a, "text_kv", False) else
        ("fwd, precision=high (split-bf16 x3 GEMMs, fp32 attention)" if getattr(a, "precision", "bf16") == "high" else "fwd"))
    law = ", R2R-CE-like text lengths (normal(32,12) in [8,80], padded)" if a.text_law else ""
    fam = ", XLM-R shape (eps 1e-5)" if getattr(a, "xlmr", False) else ""
    return (f"planner step {what}: forward_panorama+forward_navigation, B={a.batch}/GPU, V={a.views}, N={a.nodes}, "
            f"L={a.tokens}{law}{fam}, {a.x_layers} cross layers")


# ------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# ------------------------------------------------------------------------------------------------
class Clocks:
    """SM clock / throttle reasons sampled every 50 ms by a thread WHILE the timed regions run.  NVML is called in-process
    (pynvml: the library behind nvidia-smi): spawning an nvidia-smi process ten times a second means fork()ing a process
    that holds gigabytes of pinned and CUDA-mapped memory — each fork stalls the launching thread for tens of
    milliseconds, which showed up as sporadic 2-3x slow timed regions.  Falls back to the nvidia-smi command line (the
    recipe of B200_PROFILING.md) when pynvml is not importable."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.samples, self.stop, self.th = index, [], False, None
        self.nvml, self.handle, self.source = None, None, "nvidia-smi"
        try:
            import pynvml
            pynvml.nvmlInit()
            try:    # the CUDA device's own PCI address (robust to CUDA_VISIBLE_DEVICES re-numbering)
                p = torch.cuda.get_device_properties(index)
                self.handle = pynvml.nvmlDeviceGetHandleByPciBusId(f"{p.pci_domain_id:08x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0")
            except Exception:
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.nvml, self.source = pynvml, "nvml"
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        n, h = self.nvml, self.handle
        sm = n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM)
        mx = n.nvmlDeviceGetMaxClockInfo(h, n.NVML_CLOCK_SM)
        try:
            r = n.nvmlDeviceGetCurrentClocksEventReasons(h)
        except Exception:
            r = n.nvmlDeviceGetCurrentClocksThrottleReasons(h)
        act = lambda bit: "Active" if (r & bit) else "Not Active"
        return [str(sm), str(mx), act(n.nvmlClocksEventReasonHwSlowdown), act(n.nvmlClocksEventReasonHwThermalSlowdown),
                act(n.nvmlClocksEventReasonSwThermalSlowdown), act(n.nvmlClocksEventReasonSwPowerCap)]

    def _run(self):
        while not self.stop:
            try:
                if self.nvml is not None:
                    self.samples.append(self._sample_nvml())
                else:
                    out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                    self.samples.append([x.strip() for x in out.strip().split(",")])
            except Exception:
                pass
            time.sleep(0.05 if self.nvml is not None else 0.1)

    def __enter__(self):
        self.th = threading.Thread(target=self._run, daemon=True)
        self.th.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        self.th.join(timeout=6)

    def summary(self):
        sm = sorted(int(s[0]) for s in self.samples if len(s) >= 6 and s[0].isdigit())
        mx = [int(s[1]) for s in self.samples if len(s) >= 6 and s[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for s in self.samples if len(s) >= 6 for i in range(4) if s[2 + i].startswith("Active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx[0] if mx else None,
                "reasons": reasons, "samples": len(sm), "source": self.source}


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference on the host cores
# ------------------------------------------------------------------------------------------------
def _use_torch_primitives(P):
    """The reference's layers are nn.Linear (addmm) and nn.LayerNorm (vilmodel_cmt.py:24-28): time the port with those
    fused torch primitives, not with its readable ``x @ W.t() + b`` / six-op LayerNorm restatement."""
    import torch.nn.functional as F
    P._lin = lambda sd, name, x: F.linear(x, sd[name + ".weight"], sd[name + ".bias"])
    P._ln = lambda sd, name, x, eps: F.layer_norm(x, (x.shape[-1],), sd[name + ".weight"], sd[name + ".bias"], eps)


def cpu_step_time(a, mode, steps, warmup, budget_s=25.0):
    """Median step time of the oracle port of the reference on the host cores.  ``steps`` / ``warmup`` are honoured as
    long as the whole run fits ``budget_s``; otherwise they are cut and the reason is returned."""
    from oracle import planner_port as P  # test infrastructure, used here only as the timed CPU baseline
    _use_torch_primitives(P)
    cores = os.cpu_count() or 1
    try:
        cores = len(os.sched_getaffinity(0))
    except Exception:
        pass
    cfg = workload_cfg(a)
    sd = make_weights(cfg, seed=0, skip_text=False)
    # torch's CPU GEMMs do not always scale to every hardware thread of a big host: time a small forward at a few
    # thread counts and keep the fastest ("all the host threads it can use")
    cand = sorted({c for c in (cores, cores // 2, 64, 32, 16) if 1 <= c <= cores}, reverse=True)
    if len(cand) > 1:
        small = make_inputs(cfg, 4, a.views, a.nodes, a.tokens, seed=2, ragged=False)
        best = (None, 1e30)
        for c in cand:
            torch.set_num_threads(c)
            ts = []
            for _ in range(3):
                t0 = time.perf_counter()
                with torch.no_grad():
                    P.forward_navigation(sd, cfg, small["txt_embeds"], small["txt_masks"], None, small["gmap_step_ids"],
                                         small["gmap_img_fts"], small["gmap_pos_fts"], small["gmap_masks"],
                                         small["gmap_visited_masks"], small["gmap_pair_dists"])
                ts.append(time.perf_counter() - t0)
            if min(ts[1:]) < best[1]:
                best = (c, min(ts[1:]))
        cores = best[0]
    torch.set_num_threads(cores)
    inp = make_inputs(cfg, a.batch, a.views, a.nodes, a.tokens, seed=1, ragged=False, txt_law=a.text_law)
    if mode == "train":
        sd = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
        opt = torch.optim.AdamW([v for v in sd.values()], lr=1e-5)

    drop = torch_dropout_hook(cfg) if mode == "train" else None

    def step():
        if mode == "train":
            opt.zero_grad(set_to_none=True)
            pano, pm = P.forward_panorama(sd, cfg, inp["rgb_fts"], inp["dep_fts"], inp["loc_fts"], inp["nav_types"], inp["view_lens"],
                                          drop=drop)
            nav = P.forward_navigation(sd, cfg, inp["txt_embeds"], inp["txt_masks"], None, inp["gmap_step_ids"],
                                       inp["gmap_img_fts"], inp["gmap_pos_fts"], inp["gmap_masks"],
                                       inp["gmap_visited_masks"], inp["gmap_pair_dists"], drop=drop)
            loss = P.step_loss(nav["global_logits"], inp["labels"]) + (pano * pm[..., None]).sum() * 1e-3
            loss.backward()
            opt.step()
        else:
            with torch.no_grad():
                P.forward_panorama(sd, cfg, inp["rgb_fts"], inp["dep_fts"], inp["loc_fts"], inp["nav_types"], inp["view_lens"])
                P.forward_navigation(sd, cfg, inp["txt_embeds"], inp["txt_masks"], None, inp["gmap_step_ids"],
                                     inp["gmap_img_fts"], inp["gmap_pos_fts"], inp["gmap_masks"],
                                     inp["gmap_visited_masks"], inp["gmap_pair_dists"])

    t_all = time.perf_counter()
    t0 = time.perf_counter()
    step()                                   # first warm-up step (allocator, thread pool): also the cost estimate
    t_first = time.perf_counter() - t0
    n_warm, cap = 1, None
    fit = max(1, int(budget_s / max(t_first, 1e-6)) - 1)          # steps that still fit after the first one
    want_warm = max(0, warmup - 1)
    do_warm = min(want_warm, max(0, fit // 5))
    do_steps = min(steps, max(1, fit - do_warm))
    if do_warm < want_warm or do_steps < steps:
        cap = (f"requested {steps} steps / {warmup} warm-up; one step takes {t_first:.1f} s on this host, the {budget_s:.0f} s "
               f"budget fits {do_steps} timed + {1 + do_warm} warm-up")
    for _ in range(do_warm):
        step()
        n_warm += 1
    times = []
    for _ in range(do_steps):
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
    times.sort()
    med = times[len(times) // 2]
    return med, cores, len(times), n_warm, cap, time.perf_counter() - t_all


def gpu_eager_time(a, mode, dev, autocast, steps=10, warmup=3):
    """Eager-PyTorch GPU baseline: the oracle port (the reference's op sequence) with torch's own fused
    F.linear / F.layer_norm, fp32 or bf16 autocast, same workload, CUDA-event timed.  A reported baseline only."""
    from oracle import planner_port as P  # test infrastructure, used here only as a timed baseline
    _use_torch_primitives(P)
    cfg = workload_cfg(a)
    sd = {k: v.to(dev) for k, v in make_weights(cfg, seed=0, skip_text=False).items()}
    inp = {k: (v.to(dev) if isinstance(v, torch.Tensor) else v)
           for k, v in make_inputs(cfg, a.batch, a.views, a.nodes, a.tokens, seed=1, ragged=False, txt_law=a.text_law).items()}
    if mode == "train":
        sd = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
        opt = torch.optim.AdamW(list(sd.values()), lr=1e-5)

    drop = torch_dropout_hook(cfg) if mode == "train" else None

    def fwd():
        pano, pm = P.forward_panorama(sd, cfg, inp["rgb_fts"], inp["dep_fts"], inp["loc_fts"], inp["nav_types"], inp["view_lens"],
                                      drop=drop)
        nav = P.forward_navigation(sd, cfg, inp["txt_embeds"], inp["txt_masks"], None, inp["gmap_step_ids"],
                                   inp["gmap_img_fts"], inp["gmap_pos_fts"], inp["gmap_masks"],
                                   inp["gmap_visited_masks"], inp["gmap_pair_dists"], drop=drop)
        return pano, pm, nav

    def step():
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
            if mode == "train":
                opt.zero_grad(set_to_none=True)
                pano, pm, nav = fwd()
                loss = P.step_loss(nav["global_logits"].float(), inp["labels"]) + (pano.float() * pm[..., None]).sum() * 1e-3
            else:
                with torch.no_grad():
                    fwd()
        if mode == "train":
            loss.backward()
            opt.step()

    for _ in range(warmup):
        step()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def run_reference_arm(a, mode, rank, world):
    """``--impl reference``: the reference's own CPU implementation of the path (oracle port: the reference itself cannot
    travel to the GPU box) with torch's nn.Linear / nn.LayerNorm primitives, all host threads it can use.  Same ``config``,
    ``metric`` and ``unit`` as the B200 arm.  Under torchrun only rank 0 works.  The metric counts B-episode planner steps
    per second for the whole job; a host has one set of cores whatever N is, so its whole-job rate is 1 / (time of one
    B-episode step): every timed step is that bounded sample (1/N of the N-GPU job's global batch)."""
    if rank != 0:
        return
    med, cores, n, n_warm, cap, wall = cpu_step_time(a, mode, a.steps, a.warmup, budget_s=200.0)
    val = 1.0 / med
    sample = (f"{n} timed step(s) after {n_warm} warm-up, median; each step = one B={a.batch} batch of the workload"
              + (f" (1/{world} of the job's global batch: the host's whole-job rate does not depend on N)" if world > 1 else "")
              + "; oracle port of the reference with torch nn.Linear / nn.LayerNorm primitives, fp32, torch CPU AdamW")
    line = {"metric": metric_name(a), "value": val, "unit": "steps/s", "n_gpus": a.gpus, "steps": n, "warmup": n_warm,
            "steps_requested": a.steps, "warmup_requested": a.warmup, "cap": cap,
            "ms_per_step": med * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": config_dict(a, mode, world),
            "cpu_baseline": {"value": val, "unit": "steps/s", "cores": cores, "kind": "port", "sample": sample,
                             "wall_s": wall},
            "e2e": {"value": val, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# secondary workloads (SURVEY.md 8f rows N2 / N3): same timing rules, their own metric names, single GPU
# ------------------------------------------------------------------------------------------------
def _timed_events(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def _host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def run_pretrain_workload(a):
    """One pre-training iteration = one task batch (mlm, then sap, alternating as mix_ratio 1:1 of
    run_pt/r2r_pretrain_habitat.json) forward + backward + AdamW at train_batch_size 32, <= 7 viewpoints x 36 views per
    episode, <= 100 tokens, 9 language / 2 panorama / 4 cross-modal layers, train() dropout on."""
    from etpnav_b200 import lib as L
    from etpnav_b200.pretrain import B200PreTraining, PretrainTrainer
    from etpnav_b200.synth import make_traj_batch
    torch.cuda.set_device(0)
    L.require_device()
    cfg = PlannerConfig(vocab_size=30522, num_l_layers=9, num_x_layers=4, use_lang2visn_attn=True, mlm_head=True)
    model = B200PreTraining(cfg, device="cuda").train()
    sd = make_weights(cfg, seed=0)
    model.bert.load_state_dict(sd, strict=True)
    host = make_traj_batch(cfg, 32, 7, 36, 100, seed=3, ghosts=20)
    dev_batch = {k: (v.cuda() if isinstance(v, torch.Tensor) else v) for k, v in host.items()}
    tr = PretrainTrainer(model, world_size=1)
    lib = L.lib()
    lib.etp_launch_count.restype = __import__("ctypes").c_longlong
    state = {"i": 0}

    def it(batch=dev_batch):
        tr.step(batch, "mlm" if state["i"] % 2 == 0 else "sap")
        state["i"] += 1

    ms = _timed_events(it, max(2, a.steps // 2 * 2), max(4, a.warmup))
    n0 = lib.etp_launch_count()
    it(); it()
    launches = (lib.etp_launch_count() - n0) / 2

    pinned = {k: (v.pin_memory() if isinstance(v, torch.Tensor) else v) for k, v in host.items()}

    def e2e_it():   # host batch: every tensor crosses PCIe inside the timed region, the loss comes back
        d = {k: (v.cuda(non_blocking=True) if isinstance(v, torch.Tensor) else v) for k, v in pinned.items()}
        tr.step(d, "mlm" if state["i"] % 2 == 0 else "sap").item()
        state["i"] += 1
    e2e_ms = _timed_events(e2e_it, max(2, a.steps // 2 * 2), 2)
    h2d = sum(v.numel() * v.element_size() for v in host.values() if isinstance(v, torch.Tensor))
    cpu = None
    if not a.no_cpu_baseline:
        from oracle import pretrain_port as PP  # test infrastructure, used here only as the timed CPU baseline
        cores = min(_host_cores(), 32)
        torch.set_num_threads(cores)
        sdc = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
        opt = torch.optim.AdamW(list(sdc.values()), lr=5e-5, betas=(0.9, 0.98), weight_decay=0.01)
        ts = []
        for task in ("mlm", "sap", "mlm", "sap"):
            t0 = time.perf_counter()
            opt.zero_grad(set_to_none=True)
            (PP.task_mlm(sdc, cfg, host) if task == "mlm" else PP.task_sap(sdc, cfg, host)).mean().backward()
            opt.step()
            ts.append(time.perf_counter() - t0)
        med = (ts[2] + ts[3]) / 2
        cpu = {"value": 1.0 / med, "unit": "iterations/s", "cores": cores, "kind": "port",
               "sample": "one mlm + one sap iteration after one warm-up pair; oracle/pretrain_port.py fp32 autograd + torch AdamW"}
    line = {"metric": "pre-training iterations/sec (B=32, <=7 viewpoints x 36 views, <=100 tokens; mlm/sap alternating)",
            "value": 1e3 / ms, "unit": "iterations/s", "n_gpus": 1, "steps": max(2, a.steps // 2 * 2), "warmup": max(4, a.warmup),
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic",
            "config": {"workload": "GlocalTextPathCMTPreTraining iteration: fwd+bwd+AdamW, tasks mlm and sap alternating, "
                                   "train() dropout on, 9/2/4 layers, vocab 30522",
                       "view_tokens": int(host["traj_view_img_fts"].shape[0] * 36), "nodes": int(host["gmap_step_ids"].shape[1]),
                       "masked_tokens": int((host["txt_labels"] != -1).sum())},
            "e2e": {"value": 1e3 / e2e_ms, "unit": "iterations/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4},
            "gpu_launches": launches, "cpu_baseline": cpu}
    print(json.dumps(line), flush=True)


def run_packing_workload(a):
    """One packing step = ETPTrainer._nav_gmap_variable for B=64 environments whose maps EVOLVE the way GraphMap.update_graph
    makes them (tests/gmap_sim.py: one new node per step, ghosts created / merged / deleted, the all-pairs tables rebuilt
    by networkx; untimed) up to about 15 visited nodes + 50-60 ghosts.  Timed, per step, with a synchronize: the stateful
    packer (packing.GmapPacker: incremental mirror + one H2D + two launches) and the stateless pack_gmap on the same maps,
    against the oracle port of the reference's Python loops on the host."""
    import numpy as np
    from etpnav_b200 import lib as L
    from etpnav_b200 import packing
    from tests.gmap_sim import SimGraphMap     # synthetic map generator (test infrastructure), not a checker
    torch.cuda.set_device(0)
    L.require_device()
    B, grow, timed = a.batch, 6, 6     # 7 -> 14 visited nodes over the run, ~80 map rows at the end (the c3 shape)
    gms = [SimGraphMap(e, width=768, device="cuda", ghost_aug=0.0, p_node=0.03, p_ghost=0.15) for e in range(B)]
    for gm in gms:
        for _ in range(grow):
            gm.step(n_cands=7)
    pk = packing.GmapPacker("cuda")
    t_inc, t_full, t_host, closures = [], [], [], 0
    with torch.no_grad():
        for t in range(timed + 2):
            for gm in gms:
                gm.step(n_cands=7)
                closures += len(gm.graph_nx[gm.cur_vp]) > 1
            cur_vp, cur_pos, cur_ori = (list(x) for x in zip(*[gm.pose() for gm in gms]))
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = pk.pack(gms, cur_vp, cur_pos, cur_ori)
            t1 = time.perf_counter()
            torch.cuda.synchronize()
            t2 = time.perf_counter()
            ref = packing.pack_gmap(gms, cur_vp, cur_pos, cur_ori, "cuda")
            torch.cuda.synchronize()
            t3 = time.perf_counter()
            for k in ("gmap_step_ids", "gmap_visited_masks", "gmap_masks", "gmap_pos_fts", "gmap_pair_dists", "gmap_img_fts"):
                assert torch.equal(out[k], ref[k]), k          # the two packers agree bit for bit on every timed step
            if t >= 2:
                t_inc.append((t2 - t0) * 1e3); t_host.append((t1 - t0) * 1e3); t_full.append((t3 - t2) * 1e3)
    n_max = int(out["gmap_step_ids"].shape[1])
    e2e_ms, full_ms = float(np.median(t_inc)), float(np.median(t_full))
    from oracle import packing_port as PK  # test infrastructure: the reference's loops restated, timed as the CPU baseline
    sts = [PK.MapState.from_graph_map(gm) for gm in gms]
    ne = [[gm.node_embeds[v].cpu() for v in gm.node_pos] for gm in gms]
    ge = [[(gm.ghost_embeds[v][0].cpu(), gm.ghost_embeds[v][1]) for v in gm.ghost_pos] for gm in gms]
    t0 = time.perf_counter()
    PK.nav_gmap_variable(sts, [len(gm.node_pos) - 1 for gm in gms], cur_pos, cur_ori, ne, ge)
    cpu_ms = (time.perf_counter() - t0) * 1e3
    out_bytes = B * n_max * (n_max + 7) * 4 + B * n_max * 10
    n_nodes = int(np.mean([len(gm.node_pos) for gm in gms]))
    line = {"metric": f"map packs/sec (B={B} environments, up to {n_max} map rows each)", "value": 1e3 / e2e_ms, "unit": "packs/s",
            "n_gpus": 1, "steps": timed, "warmup": 2, "ms_per_step": e2e_ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64->f32", "data": "synthetic",
            "config": {"workload": "ETPTrainer._nav_gmap_variable replacement on evolving maps: every environment gains a node "
                                   "(and ghosts) between two packs",
                       "visited_nodes_mean": n_nodes, "loop_closure_steps_frac": closures / (B * (timed + 2)),
                       "stateful_packer_ms": e2e_ms, "stateful_packer_host_ms": float(np.median(t_host)),
                       "stateless_pack_gmap_ms": full_ms},
            "e2e": {"value": 1e3 / e2e_ms, "unit": "packs/s", "h2d_bytes_per_step": int(pk._last_blob.numel()),
                    "d2h_bytes_per_step": 0},
            "gpu_launches": 2,
            "roofline": {"bound": "hbm", "kernel": "gmap_pack_kernel", "achieved": None, "peak": None, "unit": "GB/s", "frac": None,
                         "traffic": None, "note": f"{out_bytes} output bytes per launch: latency-bound at this size (one CTA per environment)"},
            "cpu_baseline": {"value": 1e3 / cpu_ms, "unit": "packs/s", "cores": 1, "kind": "port",
                             "sample": "one full-size call of oracle/packing_port.py:nav_gmap_variable (the reference's Python loops)"}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------
# per array (16 MiB of float32).  At most four arrays are written and two of them (masks, logits) are small, so a dump
# stays under 64 MB.
DUMP_MAX_ELEMS = 1 << 22


def dump_outputs(path, arrays, model=None):
    """``--dump-outputs``: every array the last timed step handed its caller and, after a training step, the parameters it
    updated in place (all of them in name order), as float32 DIR/<name>.npy.  An array larger than DUMP_MAX_ELEMS is
    replaced by a fixed, seeded sample of its flattened entries (the same indices for every build at the same shape).
    The node logits are -inf at masked nodes (visited or padding): an array with -inf entries is written with 0 there,
    and DIR/<name>_masked.npy holds 1 where they were, so every file is finite (NaN and +inf are left as they are)."""
    import numpy as np
    arrays = dict(arrays)
    if model is not None:
        arrays["params"] = torch.cat([p.detach().flatten() for _, p in sorted(model.named_parameters())])
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach().float()
        if t.numel() > DUMP_MAX_ELEMS:
            idx = torch.randint(0, t.numel(), (DUMP_MAX_ELEMS,), generator=torch.Generator().manual_seed(0)).sort().values
            t = t.flatten()[idx.to(t.device)]
        masked = t == float("-inf")
        if bool(masked.any()):
            np.save(os.path.join(path, name + "_masked.npy"), masked.float().cpu().numpy())
            t = t.masked_fill(masked, 0.0)
        np.save(os.path.join(path, name + ".npy"), t.cpu().numpy())


def _latest_profile(prefix_glob):
    import glob
    c = sorted(glob.glob(os.path.join(ROOT, "profiles", prefix_glob)))
    return c[-1] if c else None


def main():
    # One hardware work queue per CUDA stream: the step uses three streams (compute, the trainer's update stream, the
    # input stager's copy stream).  With the default of 8 connections two of them can share a queue, and then the next
    # step's host->device copy sits behind the update stream's pending event wait (observed: e2e 94-112 steps/s in some
    # processes, 178-183 in others, same box, the copy alone at 55 GB/s in both).  Must be set before the CUDA context exists.
    os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
    a = parse()
    # train mode's dropout seed stream starts at torch.initial_seed() (plus the rank): fixed, so that two runs with the same
    # arguments compute the same step (--dump-outputs)
    torch.manual_seed(0)
    if a.workload == "pretrain":
        return run_pretrain_workload(a)
    if a.workload == "packing":
        return run_packing_workload(a)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    from etpnav_b200 import planner as PL
    mode = a.mode or ("train" if hasattr(PL.B200Planner, "make_trainer") else "fwd")
    if a.impl == "reference":
        run_reference_arm(a, mode, rank, world)
        return

    from etpnav_b200 import lib as L
    from etpnav_b200.pipeline import HostBatchStager, bind_to_gpu_numa
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_numa(local)      # before any pinned allocation: the staging blob lives next to this GPU's PCIe root
    if world > 1:
        import torch.distributed as dist
        if a.nccl_max_ctas > 0:
            os.environ["NCCL_MAX_CTAS"] = str(a.nccl_max_ctas)
        # NCCL prints its version banner on stdout at first use: keep stdout for the one JSON line
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.all_reduce(torch.zeros(1, device=dev))
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
    L.require_device()

    cfg = workload_cfg(a)
    model = PL.B200Planner(cfg, device=dev)
    model.load_state_dict(make_weights(cfg, seed=0), strict=True)
    B, V, N, Lt = a.batch, a.views, a.nodes, a.tokens
    host = make_inputs(cfg, B, V, N, Lt, seed=100 + rank, ragged=False, txt_law=a.text_law)
    keys_pano = ["rgb_fts", "dep_fts", "loc_fts", "nav_types", "view_lens"]
    keys_nav = ["txt_embeds", "txt_masks", "gmap_step_ids", "gmap_img_fts", "gmap_pos_fts", "gmap_masks",
                "gmap_visited_masks", "gmap_pair_dists"]
    step_keys = keys_pano + keys_nav + ["labels"]
    resident = {k: host[k].to(dev) for k in step_keys}
    # host side of the e2e leg: ONE pinned blob per step (txt_embeds staged as bf16: the kernels' first act on it is that cast)
    stager = HostBatchStager(dev, slots=2, bf16_keys=() if a.precision == "high" else ("txt_embeds",))
    # (with --text-kv the instruction stays on the device for the whole episode, as forward_txt's output does in the
    # reference: it is not a per-step input any more)
    blob, blob_meta = stager.pack({k: host[k] for k in step_keys if not (a.text_kv and mode == "fwd" and k == "txt_embeds")})
    h2d_bytes = int(blob_meta[2])
    logits_host = torch.empty(B, N, dtype=torch.float32).pin_memory()
    d2h_bytes = logits_host.numel() * 4
    last = {}       # what the latest step handed its caller (--dump-outputs)

    if mode == "train":
        model.train()
        if a.peer_ctas > 0:
            os.environ["ETP_PEER_CTAS"] = str(a.peer_ctas)
        trainer = model.make_trainer(lr=1e-5, world_size=world, grad_comm=a.grad_comm, comm_sms=a.comm_sms)

        def step(d):
            # training-loop form of the step: the compute stream returns once the navigation buckets are updated, the
            # panorama buckets finish under the next step's first GEMM; every timed region ends with trainer.join()
            last["global_logits"] = trainer.step(d, pipelined=True)
            return last["global_logits"]

        step_done = trainer.join
    else:
        step_done = lambda: None
        model.eval().set_precision(a.precision)
        text_kv = None
        if a.text_kv:   # once per episode, like forward_txt: not part of the per-step path
            with torch.no_grad():
                text_kv = model.encode_text_kv(resident["txt_embeds"])

        def step(d):
            with torch.no_grad():
                last["pano_embeds"], last["pano_masks"] = model.forward_panorama(*[d[k] for k in keys_pano])
                out = model.forward_navigation(text_kv if text_kv is not None else d["txt_embeds"], d["txt_masks"], None,
                                               d["gmap_step_ids"], d["gmap_img_fts"], d["gmap_pos_fts"], d["gmap_masks"],
                                               d["gmap_visited_masks"], d["gmap_pair_dists"])
            last.update(out)
            return out["global_logits"]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(steps):
            fn()
        step_done()          # nothing of the last step is left running outside the timed region
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    for _ in range(max(3, a.warmup)):
        step(resident)
    peer_runtime_fallback = None
    if world > 1 and mode == "train" and trainer.grad_comm == "peer":
        # a flag wait of the peer-memory update that gave up (a rank far behind, a mapping that does not behave) would make
        # every later number meaningless: all ranks then agree to redo the warm-up on the NCCL path and say so
        trainer.join()
        err = torch.tensor([trainer.peer_error()], device=dev)
        dist.all_reduce(err, op=dist.ReduceOp.MAX)
        if int(err.item()) != 0:
            peer_runtime_fallback = f"peer flag wait timed out during warm-up (code {int(err.item())}): NCCL path used instead"
            trainer = model.make_trainer(lr=1e-5, world_size=world, grad_comm="fp32", comm_sms=a.comm_sms)
            step_done = trainer.join
            for _ in range(max(3, a.warmup)):
                step(resident)
    lib = L.lib()
    lib.etp_launch_count.restype = __import__("ctypes").c_longlong
    n0 = lib.etp_launch_count()
    clk = Clocks(local)
    clk.__enter__()   # sampled across the timed regions below (value, e2e): all under load
    total_ms = timed(lambda: step(resident), a.steps)
    launches = lib.etp_launch_count() - n0
    if a.dump_outputs and rank == 0:     # before any later pass runs another step
        dump_outputs(a.dump_outputs, last, model if mode == "train" else None)
    ms_per_step = total_ms / a.steps
    value = world / (ms_per_step * 1e-3)

    # host side of one step: time to ENQUEUE it with an empty launch queue (no synchronisation inside): if this is close
    # to ms_per_step the step is launch-bound on the host, not GPU-bound
    host_ms = []
    for _ in range(5):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        step(resident)
        host_ms.append((time.perf_counter() - t0) * 1e3)
    torch.cuda.synchronize()
    host_ms.sort()
    host_enqueue_ms = host_ms[len(host_ms) // 2]

    # end-to-end: host blob -> ONE H2D copy -> step -> D2H logits, through the public API.  Every step's inputs cross PCIe
    # inside the timed region; the copy of step t+1 is issued on a side stream while step t computes
    # (etpnav_b200.pipeline.HostBatchStager: two device slots), the compute stream waits on its event.
    def e2e_run(n):
        stager.submit(blob, blob_meta)
        for i in range(n):
            d = stager.get()
            if i + 1 < n:
                stager.submit(blob, blob_meta)      # next step's inputs start crossing PCIe now
            lg = step(d)
            logits_host.copy_(lg, non_blocking=True)

    def h2d_alone_gbps():
        """The blob's host -> device copy with nothing else on the GPU (GB/s): tells a slow / contended host link (this
        number is low too) from a copy starved by the overlapped compute (this number is fine, e2e is not)."""
        dst = torch.empty(h2d_bytes, dtype=torch.uint8, device=dev)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(4):
            dst.copy_(blob[:h2d_bytes], non_blocking=True)
        e1.record()
        torch.cuda.synchronize()
        return 4 * h2d_bytes / (e0.elapsed_time(e1) * 1e-3) / 1e9

    def e2e_run_serial(n):
        """The other staging policy: the blob is copied on the COMPUTE stream at the start of its own step (no overlap, no
        second stream).  Costs the copy time per step but cannot be delayed by anything; reported next to the overlapped
        policy, the better of the two is the e2e value (some processes of this pool see the overlapped copy starve)."""
        dst = torch.empty(h2d_bytes, dtype=torch.uint8, device=dev)
        ents, extra, _ = blob_meta
        for _ in range(n):
            dst.copy_(blob[:h2d_bytes], non_blocking=True)
            d = dict(extra)
            for k, off, nbytes, dt, shape in ents:
                d[k] = dst[off:off + nbytes].view(dt).view(shape)
            lg = step(d)
            logits_host.copy_(lg, non_blocking=True)

    h2d_before = h2d_alone_gbps()
    e2e_run(3)
    e2e_ms_overlap = timed(lambda: e2e_run(a.steps), 1) / a.steps
    # one more overlapped pass with a timing event on either side of every copy: how long the copies themselves took under
    # the step (ms, min / median / max) — a starved copy shows here, a late one does not
    stager.trace = []
    ref_ev = torch.cuda.Event(enable_timing=True)
    ref_ev.record()
    e2e_run(min(a.steps, 10))
    torch.cuda.synchronize()
    dur = sorted(t0.elapsed_time(t1) for t0, t1 in stager.trace)
    start = [ref_ev.elapsed_time(t0) for t0, _ in stager.trace]
    copy_trace = {"copy_ms_min_med_max": [round(dur[0], 3), round(dur[len(dur) // 2], 3), round(dur[-1], 3)],
                  "copy_start_ms": [round(x, 2) for x in start]}
    stager.trace = None
    e2e_run_serial(2)
    e2e_ms_serial = timed(lambda: e2e_run_serial(a.steps), 1) / a.steps
    e2e_ms = min(e2e_ms_overlap, e2e_ms_serial)
    e2e_val = world / (e2e_ms * 1e-3)
    h2d_after = h2d_alone_gbps()
    clk.__exit__()

    # sustained: the same step for >= 3 s (power / clocks settle on a long region; the 20-step figure is a 0.1 s burst)
    soak = None
    if not a.no_soak:
        n_soak = int(min(4000, max(a.steps, 3000.0 / ms_per_step + 1)))
        clk2 = Clocks(local)
        clk2.__enter__()
        soak_ms = timed(lambda: step(resident), n_soak)
        clk2.__exit__()
        soak = {"ms_per_step": soak_ms / n_soak, "value": world / (soak_ms / n_soak * 1e-3), "steps": n_soak,
                "seconds": soak_ms * 1e-3, "clocks": clk2.summary()}

    # roofline of the dominant kernel (tcgen05 GEMM): profiled pass with per-launch CUDA events
    import ctypes as C
    lib.etp_prof_gemm_enable(1)
    torch.cuda.synchronize()
    prof_steps = min(a.steps, 5)
    for _ in range(prof_steps):
        step(resident)
    torch.cuda.synchronize()
    buf = C.create_string_buffer(1 << 20)
    lib.etp_prof_report.argtypes = [C.c_char_p, C.c_size_t]
    L._check(lib.etp_prof_report(buf, len(buf)), "etp_prof_report")
    lib.etp_prof_gemm_enable(0)
    g_ms, g_fl, g_n = 0.0, 0.0, 0
    rows = []
    for ln in buf.value.decode().splitlines():
        cnt, ms, fl, name, tag = (ln.split("\t") + [""])[:5]
        rows.append((int(cnt), float(ms), float(fl), name, tag))
        if float(fl) > 0:
            g_ms += float(ms); g_fl += float(fl); g_n += int(cnt)
    if a.kernel_report and rank == 0:
        tot = sum(r[1] for r in rows) or 1.0
        with open(a.kernel_report, "w") as f:
            f.write(f"# per-kernel CUDA-event time over {prof_steps} profiled step(s) of: {workload_name(a, mode)}\n")
            f.write("# count/step\tus/step\tshare\tavg_us\tTFLOP/s\tkernel\ttag\n")
            for cnt, ms, fl, name, tag in sorted(rows, key=lambda r: -r[1]):
                tf = fl / (ms * 1e-3) / 1e12 if fl > 0 and ms > 0 else 0.0
                f.write(f"{cnt / prof_steps:.1f}\t{ms * 1e3 / prof_steps:.1f}\t{ms / tot * 100:.1f}%\t{ms * 1e3 / cnt:.1f}\t{tf:.0f}\t{name}\t{tag}\n")
            f.write(f"# total {tot * 1e3 / prof_steps:.1f} us/step (events serialise the launches: PDL overlap is off in this pass)\n")
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    # the GEMMs are event-timed one launch at a time inside a sub-second region at full clock: burst conditions, so the
    # denominator is the BURST bf16 peak; the fraction of the sustained (power-capped, 4 s back-to-back) peak is given too
    peak = peaks.get("bf16_tflops", 1600.0)
    peak_sus = peaks.get("bf16_tflops_sustained", 1400.0)
    peak_src = ("measured (MEASURED_PEAKS.json bf16_tflops, burst: kernels event-timed alone in a short region)" if peaks
                else "fallback 1.6 PF burst / 1.4 PF sustained (B200_PROFILING.md)")
    achieved = (g_fl / (g_ms * 1e-3)) / 1e12 if g_ms > 0 else 0.0
    fl = step_flops(cfg, B, V, N, Lt)
    traffic, traffic_note = None, "no ncu summary found under profiles/"
    try:   # mean dram__bytes_read + dram__bytes_write per GEMM launch over one captured step (profiles/summarize_ncu.py)
        tpath = _latest_profile("r0*_gemm_traffic.json")
        tj = json.load(open(tpath))
        traffic = tj["mean_dram_bytes_per_launch"]
        traffic_note = (f"mean over {tj['launches']} GEMM launches of one c3 train step captured with ncu "
                        f"({os.path.relpath(tpath, ROOT)}); tensor pipe active {tj['tensor_pipe_active_pct_time_weighted']:.1f} % "
                        "time-weighted over those launches")
    except Exception:
        pass
    step_tf = (fl["step_fwd"] * (3 if mode == "train" else 1)) / (ms_per_step * 1e-3) / 1e12
    roof = {"bound": "tensor", "kernel": "gemm_tcgen05_kernel", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
            "frac": achieved / peak, "traffic": traffic, "traffic_note": traffic_note,
            "peak_source": peak_src, "frac_of_sustained_peak": achieved / peak_sus,
            "gemm_launches_per_step": g_n / prof_steps, "gemm_ms_per_step": g_ms / prof_steps,
            "gemm_share_of_step": (g_ms / prof_steps) / ms_per_step,
            "step_model_tflops": step_tf, "step_frac_of_burst_peak": step_tf / peak}

    # data-parallel self-check (N > 1): ONE extra step with identical data, weights and dropout seed on every rank.  The
    # bucketed, event-triggered all-reduce must then return N x the local gradient: g_reduced / N is compared with the
    # gradient of the same step taken WITHOUT any collective, and the ranks' updated parameters with each other.  A bucket
    # reduced before its gradients were final shows up as an O(1) relative error; summation-order noise (fp32 atomics in
    # the weight-gradient / LayerNorm kernels) is ~1e-6.
    dp = None
    if world > 1 and mode == "train" and not a.no_dp_check:
        same = {k: v.to(dev) for k, v in make_inputs(cfg, B, V, N, Lt, seed=999, ragged=False, txt_law=a.text_law).items()
                if isinstance(v, torch.Tensor)}
        sd0 = make_weights(cfg, seed=0)
        res = []
        for w_ in (world, 1):
            m2 = PL.B200Planner(cfg, device=dev)
            m2.load_state_dict(sd0, strict=True)
            m2.train()
            m2.set_dropout_seed(777)
            t2 = m2.make_trainer(lr=1e-5, world_size=w_, grad_comm=a.grad_comm, comm_sms=a.comm_sms)
            if getattr(t2, "_peer", None) is not None:
                t2._peer_write_reduced = 1     # the owner leaves the summed gradient in its own buffer: that is what is checked
            m2.set_dropout_seed(777)
            t2.step(same, keep_grads=True)
            torch.cuda.synchronize()
            if w_ > 1:
                owned, perr, dp_path = t2.owned_ranges(), t2.peer_error(), t2.grad_comm + (
                    f" (peer unavailable: {t2.peer_fallback})" if t2.peer_fallback else "")
            res.append((m2._direct_grad[t2.lo:t2.hi].clone() * (1.0 / w_), m2._flat[t2.lo:t2.hi].clone()))
            del m2, t2
        (g_dp, p_dp), (g_1, p_1) = res
        gmax = g_1.abs().max().clamp_min(1e-30)
        # peer mode: a rank holds the reduced gradient of the sub-slices it owns (the ranks together cover the buffer)
        gerr = torch.stack([(g_dp[x:y] - g_1[x:y]).abs().max() for x, y in owned if y > x]).max()
        stats = torch.stack([gerr / gmax, (p_dp - p_1).abs().max()]).double()
        pmin, pmax = p_dp.clone(), p_dp.clone()
        dist.all_reduce(pmin, op=dist.ReduceOp.MIN)
        dist.all_reduce(pmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
        dp = {"dp_check_grad_max_rel": float(stats[0]), "dp_check_max_abs": float(stats[1]),
              "dp_check_cross_rank_param_max_abs": float((pmax - pmin).abs().max()), "peer_wait_error": perr,
              "update_path_checked": dp_path,
              "what": "one step, identical data / weights / dropout seed on all ranks: all-reduced gradient / N vs the "
                      "collective-free gradient (max |d| / max |g|), updated parameters vs the collective-free step and across ranks"}

    if rank == 0:
        cpu = None
        if world == 1 and not a.no_cpu_baseline:
            med, cores, n, n_warm, cap, wall = cpu_step_time(a, mode, steps=3, warmup=1, budget_s=25.0)
            cpu = {"value": 1.0 / med, "unit": "steps/s", "cores": cores, "kind": "port",
                   "sample": f"median of {n} full-size step(s) after {n_warm} warm-up; oracle/planner_port.py with torch nn.Linear / "
                             "nn.LayerNorm primitives, fp32, torch CPU"}
        eager = None
        if world == 1 and not a.no_gpu_eager:
            ms32 = gpu_eager_time(a, mode, dev, autocast=False)
            ms16 = gpu_eager_time(a, mode, dev, autocast=True)
            eager = {"fp32_steps_per_s": 1e3 / ms32, "bf16_autocast_steps_per_s": 1e3 / ms16, "unit": "steps/s",
                     "speedup_vs_fp32_eager": (1e3 / ms_per_step) / (1e3 / ms32),
                     "speedup_vs_bf16_autocast_eager": (1e3 / ms_per_step) / (1e3 / ms16),
                     "what": "oracle port of the reference, eager PyTorch on this GPU (F.linear/F.layer_norm, torch AdamW): the "
                             "'reference GPU eager' step of the north_star's >= 10x target (fp32 = its eval path, autocast = its "
                             "training path, ss_trainer_ETP.py:502)"}
        line = {"metric": metric_name(a), "value": value, "unit": "steps/s", "n_gpus": world, "steps": a.steps,
                "warmup": max(3, a.warmup), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": ("bf16x3 (split) / f32" if (mode == "fwd" and a.precision == "high") else "bf16"),
                "data": "synthetic",
                "config": config_dict(a, mode, world),
                "e2e": {"value": e2e_val, "unit": "steps/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                        "ms_per_step": e2e_ms, "copies_per_step": {"h2d": 1, "d2h": 1},
                        "staging": "one pinned blob per step (all input tensors, 256-byte aligned)"
                                   + ("" if a.precision == "high" else ", txt_embeds as bf16"),
                        "policy": "overlapped" if e2e_ms_overlap <= e2e_ms_serial else "serial",
                        "ms_per_step_by_policy": {"overlapped (copy of step t+1 on a side stream under step t)": e2e_ms_overlap,
                                                  "serial (copy on the compute stream at the start of its step)": e2e_ms_serial},
                        "overlapped_copy_trace": copy_trace, "numa": numa, "h2d_alone_gbps": [round(h2d_before, 2), round(h2d_after, 2)]},
                "gpu_launches": int(launches), "host_enqueue_ms_per_step": host_enqueue_ms, "clocks": clk.summary(),
                "roofline": roof, "cpu_baseline": cpu}
        if soak:
            line["sustained"] = soak
        if dp:
            line["dp_check"] = dp
        if world > 1 and mode == "train":
            line["dp_update"] = {"requested": a.grad_comm, "effective": trainer.grad_comm,
                                 "peer_fallback": trainer.peer_fallback or peer_runtime_fallback,
                                 "peer_wait_error": trainer.peer_error()}
        if eager:
            line["gpu_eager_baseline"] = eager
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
