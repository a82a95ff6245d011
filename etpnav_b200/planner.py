"""Drop-in host module for the ETPNav cross-modal planner on B200.

``B200Planner`` exposes the three methods ``ETP.forward`` calls on ``self.vln_bert``
(vlnce_baselines/models/Policy_ViewSelection_ETP.py:167,346,352-357) with the reference's positional
signatures and return structures, and a ``state_dict()`` with the reference's 307 keys
(vlnce_baselines/models/etp/vilmodel_cmt.py:663-750; SURVEY.md Appendix B), so reference checkpoints load
unchanged.  All arithmetic runs in the sm_100a kernels of ``libetpnav_b200.so`` through the step-level C
ABI (include/etpnav_b200.h); PyTorch only owns memory, streams and the autograd graph.  There is no
PyTorch/CPU fallback: without the library or a B200 the methods raise.

Numerics: GEMM operands are bf16 (fp32 accumulation in TMEM); the residual stream, LayerNorm, softmax,
biases and all reductions are fp32.  fp32 master parameters live in one flat buffer (``layout.py``) whose
bf16 image is refreshed whenever a parameter changes.
"""
import ctypes as C

import torch
import torch.nn as nn

from . import lib as _L
from .config import PlannerConfig
from .layout import FlatLayout

p_void, i32, f32 = C.c_void_p, C.c_int32, C.c_float


# ----------------------------------------------------------------------------------------------------
# ctypes mirrors of the step-level structs in include/etpnav_b200.h
# ----------------------------------------------------------------------------------------------------
class LayerWeights(C.Structure):
    _fields_ = [(n, p_void) for n in (
        "xq_w", "xq_b", "xkv_w", "xkv_b", "xo_w", "xo_b", "xln_g", "xln_b",
        "sqkv_w", "sqkv_b", "so_w", "so_b", "sln_g", "sln_b",
        "f1_w", "f1_b", "f2_w", "f2_b", "fln_g", "fln_b")]


class NavWeights(C.Structure):
    _fields_ = [("num_x_layers", i32), ("ln_eps", f32), ("layers", C.POINTER(LayerWeights))] + [
        (n, p_void) for n in ("pos_w", "pos_b", "pos_g", "pos_bb", "step_emb", "sprel_w", "sprel_b",
                              "sap0_w", "sap0_b", "sap_g", "sap_bb", "sap4_w", "sap4_b", "xkv_all_w", "xkv_all_b")]


class Dropout(C.Structure):
    """``etp_dropout``: seed + probabilities of one step-level call (train() mode)."""
    _fields_ = [("seed", C.c_uint64), ("p_hidden", f32), ("p_attn", f32), ("p_head", f32)]


class NavInputs(C.Structure):
    _fields_ = [("B", i32), ("N", i32), ("L", i32)] + [
        (n, p_void) for n in ("txt_embeds", "txt_masks", "gmap_step_ids", "gmap_img_fts", "gmap_pos_fts",
                              "gmap_masks", "gmap_visited_masks", "gmap_pair_dists")] + [
        ("dropout", C.POINTER(Dropout)), ("layer_done_events", C.POINTER(p_void)), ("txt_embeds_bf16", p_void),
        ("txt_kv_all", p_void), ("txt_kv_rows", p_void), ("txt_kv_batch", i32),
        ("side_sm_reserve", i32), ("img_ready_event", p_void), ("img_grad_event", p_void), ("txt_kv_grad", p_void)]


class PanoLayerWeights(C.Structure):
    _fields_ = [(n, p_void) for n in ("in_w", "in_b", "out_w", "out_b", "l1_w", "l1_b", "l2_w", "l2_b",
                                      "n1_g", "n1_b", "n2_g", "n2_b")]


class PanoWeights(C.Structure):
    _fields_ = [("num_pano_layers", i32), ("layer_eps", f32), ("layers", C.POINTER(PanoLayerWeights))] + [
        (n, p_void) for n in ("img_w", "img_b", "dep_w", "dep_b", "loc_w", "loc_b", "img_g", "img_bb", "dep_g",
                              "dep_bb", "loc_g", "loc_bb", "out_g", "out_bb", "nav_emb", "tok_emb1", "fin_g", "fin_b")]


class PanoInputs(C.Structure):
    _fields_ = [("B", i32), ("V", i32)] + [(n, p_void) for n in ("rgb_fts", "dep_fts", "loc_fts", "nav_types", "view_lens")] + [
        ("dropout", C.POINTER(Dropout)), ("layer_done_events", C.POINTER(p_void))]


class TxtWeights(C.Structure):
    _fields_ = [("num_l_layers", i32), ("ln_eps", f32), ("layers", C.POINTER(LayerWeights))] + [
        (n, p_void) for n in ("word_emb", "pos_emb", "type_emb0", "emb_g", "emb_b")]


_declared = False


def _declare():
    global _declared
    if _declared:
        return
    L = _L.lib()
    L.etp_nav_saved_bytes.restype = C.c_size_t
    L.etp_nav_saved_bytes.argtypes = [i32] * 5
    L.etp_nav_kv_saved_bytes.restype = C.c_size_t
    L.etp_nav_kv_saved_bytes.argtypes = [i32] * 5
    L.etp_text_kv_bwd_work_bytes.restype = C.c_size_t
    L.etp_text_kv_bwd_work_bytes.argtypes = [i32] * 3
    L.etp_backward_text_kv.argtypes = [C.POINTER(NavWeights), C.POINTER(NavWeights), p_void, p_void, i32, i32, p_void, p_void,
                                       p_void, p_void]
    L.etp_pano_saved_bytes.restype = C.c_size_t
    L.etp_pano_saved_bytes.argtypes = [i32] * 4
    L.etp_txt_saved_bytes.restype = C.c_size_t
    L.etp_txt_saved_bytes.argtypes = [i32] * 4
    L.etp_forward_navigation.argtypes = [C.POINTER(NavWeights), C.POINTER(NavInputs), p_void, p_void, p_void,
                                         C.c_size_t, i32, p_void]
    L.etp_forward_panorama.argtypes = [C.POINTER(PanoWeights), C.POINTER(PanoInputs), p_void, p_void, p_void,
                                       C.c_size_t, i32, p_void]
    L.etp_forward_txt.argtypes = [C.POINTER(TxtWeights), p_void, p_void, i32, i32, p_void, p_void, C.c_size_t, i32,
                                  p_void, C.POINTER(Dropout)]
    for fn in ("etp_nav_bwd_work_bytes",):
        getattr(L, fn).restype = C.c_size_t
        getattr(L, fn).argtypes = [i32] * 4
    for fn in ("etp_pano_bwd_work_bytes", "etp_txt_bwd_work_bytes"):
        getattr(L, fn).restype = C.c_size_t
        getattr(L, fn).argtypes = [i32] * 2
    L.etp_backward_navigation.argtypes = [C.POINTER(NavWeights), C.POINTER(NavWeights), C.POINTER(NavInputs), p_void,
                                          p_void, p_void, C.c_size_t, p_void, C.c_size_t, p_void, p_void, p_void]
    L.etp_backward_panorama.argtypes = [C.POINTER(PanoWeights), C.POINTER(PanoWeights), C.POINTER(PanoInputs), p_void,
                                        p_void, p_void, C.c_size_t, p_void, C.c_size_t, p_void, p_void, p_void]
    L.etp_backward_txt.argtypes = [C.POINTER(TxtWeights), C.POINTER(TxtWeights), p_void, p_void, i32, i32, p_void, p_void,
                                   C.c_size_t, p_void, C.c_size_t, p_void, C.POINTER(Dropout)]
    # high-precision (split-bf16 x3) inference mode
    L.etp_encode_text_kv.argtypes = [C.POINTER(NavWeights), p_void, p_void, i32, i32, p_void, p_void, p_void]
    L.etp_split3.argtypes = [p_void, p_void, C.c_int64, i32, i32, p_void]
    L.etp_hp_nav_work_bytes.restype = C.c_size_t
    L.etp_hp_nav_work_bytes.argtypes = [i32] * 4
    for fn in ("etp_hp_pano_work_bytes", "etp_hp_txt_work_bytes"):
        getattr(L, fn).restype = C.c_size_t
        getattr(L, fn).argtypes = [i32] * 2
    L.etp_forward_navigation_hp.argtypes = [C.POINTER(NavWeights), C.POINTER(NavInputs), p_void, p_void, p_void, C.c_size_t,
                                            p_void]
    L.etp_forward_panorama_hp.argtypes = [C.POINTER(PanoWeights), C.POINTER(PanoInputs), p_void, p_void, p_void, C.c_size_t,
                                          p_void]
    L.etp_forward_txt_hp.argtypes = [C.POINTER(TxtWeights), p_void, p_void, i32, i32, p_void, p_void, C.c_size_t, p_void]
    _declared = True


class _TextKVGrad:
    """Gradient side of a training ``TextKV`` handle, shared by every indexed copy of it: the rollout's fp32 dK|dV
    accumulator ``[B0 * L, X * 1536]`` and whether its backward has run.  (It holds no autograd tensor, so the backward
    node that owns it forms no reference cycle.)"""

    def __init__(self, acc):
        self.acc, self.done = acc, False


class TextKV:
    """Episode-level handle of the instruction's key|value projections for ALL cross-modal layers
    (``B200Planner.encode_text_kv``): bf16 ``[B0 * L, X * 1536]``, computed ONCE per episode instead of at every step
    of every layer (the reference recomputes them although ``txt_embeds`` is constant over the episode,
    vilmodel_cmt.py:326-328).  Pass it to ``forward_navigation`` in place of ``txt_embeds``.
    Indexing it like the trainer indexes ``all_txt_embeds[not_done_index]`` (ss_trainer_ETP.py:819-821) keeps the cache
    and records the surviving episodes as a row map — no data moves.

    A training handle (made with gradients wanted) also carries ``grad`` (the rollout's dK|dV accumulator) and ``token``,
    the autograd output of the encoding: every navigation step that reads the handle hangs off it, and after the last of
    their backwards one node turns the accumulator into the key|value weight gradient and d ``txt_embeds``."""

    def __init__(self, kv_all, batch, length, rows=None, grad=None, token=None):
        self.kv_all, self.batch, self.length, self.rows = kv_all, batch, length, rows
        self.grad, self.token = grad, token

    def __len__(self):
        return self.batch if self.rows is None else int(self.rows.numel())

    @property
    def shape(self):
        return (len(self), self.length, 768)

    def __getitem__(self, idx):
        dev = self.kv_all.device
        base = torch.arange(self.batch, device=dev, dtype=torch.int32) if self.rows is None else self.rows
        if not torch.is_tensor(idx):
            idx = torch.as_tensor(idx, device=dev)
        idx = idx.to(dev)
        rows = base[idx] if idx.dtype == torch.bool else base[idx.long()]
        return TextKV(self.kv_all, self.batch, self.length, rows.to(torch.int32).contiguous(), self.grad, self.token)


class _Holder(nn.Module):
    """Anonymous container used to reproduce the reference's dotted parameter names."""


def _f32c(t):
    return t.detach().float().contiguous()


def _txtc(t):
    """txt_embeds as the navigation kernels take it: bf16 stays bf16 (no cast kernel), everything else becomes fp32."""
    return t.detach().contiguous() if t.dtype == torch.bfloat16 else _f32c(t)


class B200Planner(nn.Module):
    """Replacement for ``GlocalTextPathNavCMT`` (vilmodel_cmt.py:663)."""

    def __init__(self, config: PlannerConfig, device="cuda"):
        super().__init__()
        self.config = config
        self.layout = FlatLayout(config)
        dev = torch.device(device)
        flat = torch.zeros(self.layout.total, dtype=torch.float32, device=dev)
        self._build_tree(flat)
        self._reset_parameters()
        self._cache_key = None
        self._structs = None
        self._bf16_fresh = False
        self._grad_structs = {}
        self._direct_grad = None      # PlannerTrainer: flat fp32 gradient buffer the backward accumulates into
        self._tok_scratch = None      # PlannerTrainer without the txt group: sink of the token-type row-1 gradient
        self._anchor = torch.zeros(1, device=dev, requires_grad=True)
        self._layer_events = None  # PlannerTrainer (world > 1): cudaEvent_t per x-layer, recorded by the nav backward
        self._drop_base = None   # dropout seed stream: base (torch.initial_seed() unless set) + call counter
        self._drop_calls = 0
        self.precision = "bf16"  # "bf16" | "high" (set_precision): split-bf16 x3 GEMMs + fp32 attention, inference only
        self._flat_hp, self._structs_hp, self._hp_key = None, None, None
        if config.fix_lang_embedding:  # vilmodel_cmt.py:675-679
            for n, p in self.named_parameters():
                if n.startswith("embeddings.") or n.startswith("lang_encoder."):
                    p.requires_grad = False
        if config.fix_pano_embedding:  # vilmodel_cmt.py:680-682
            for n, p in self.named_parameters():
                if n.startswith("img_embeddings."):
                    p.requires_grad = False

    # ------------------------------------------------------------------ parameters / flat storage
    def _build_tree(self, flat):
        self._flat = flat
        self._flat_bf16 = torch.empty(self.layout.total, dtype=torch.bfloat16, device=flat.device)
        self._pmap = {}
        for name, (off, numel, shape) in self.layout.entries.items():
            parts = name.split(".")
            mod = self
            for part in parts[:-1]:
                if not hasattr(mod, part):
                    mod.add_module(part, _Holder())
                mod = getattr(mod, part)
            p = nn.Parameter(flat[off:off + numel].view(shape))
            mod.register_parameter(parts[-1], p)
            self._pmap[name] = p

    def _reset_parameters(self):
        """HF ``_init_weights`` semantics (SURVEY.md A.5): N(0, 0.02) weights, zero biases, LayerNorm (1, 0)."""
        with torch.no_grad():
            for name, p in self._pmap.items():
                is_ln = ("LayerNorm" in name or "layer_norm" in name or ".norm" in name
                         or name.startswith("global_encoder.gmap_pos_embeddings.1")
                         or name.startswith("global_sap_head.net.2"))
                if is_ln:
                    p.fill_(1.0 if name.endswith("weight") else 0.0)
                elif name.endswith("bias"):
                    p.zero_()
                else:
                    p.normal_(0.0, 0.02)
            self._pmap["embeddings.word_embeddings.weight"][0].zero_()

    def _apply(self, fn, recurse=True):
        out = super()._apply(fn, recurse)
        # .to()/.cuda()/.float() re-materialise every parameter separately: re-pack them into one flat buffer
        first = next(iter(self._pmap.values()))
        if first.data_ptr() != self._flat.data_ptr() + 4 * self.layout.offset(next(iter(self._pmap))):
            flat = torch.zeros(self.layout.total, dtype=torch.float32, device=first.device)
            for name, (off, numel, shape) in self.layout.entries.items():
                p = self._pmap[name]
                flat[off:off + numel].copy_(p.data.reshape(-1).float())
                p.data = flat[off:off + numel].view(shape)
            self._flat = flat
            self._flat_bf16 = torch.empty(self.layout.total, dtype=torch.bfloat16, device=flat.device)
            self._cache_key = None
            self._structs = None
        return out

    def load_state_dict(self, *a, **kw):
        out = super().load_state_dict(*a, **kw)
        self._bf16_fresh = False
        self._cache_key = None
        return out

    def _flat_is_intact(self):
        base = self._flat.data_ptr()
        for name, (off, _, _) in self.layout.entries.items():
            if self._pmap[name].data_ptr() != base + 4 * off:
                return False
        return True

    def _refresh_cache(self):
        """Re-cast the flat fp32 parameters to bf16 when any parameter changed (optimizer step, load)."""
        key = self._version_key()
        if key == self._cache_key and self._structs is not None:
            # nothing was written through torch since the image was made; the fused AdamW (PlannerTrainer) rewrites the
            # flat buffer and its bf16 image together without bumping versions, and re-records the key it saw
            if self.precision == "high":
                self._refresh_hp(key)
            return
        if not self._flat.is_cuda:
            raise _L.EtpError("B200Planner parameters must live on a CUDA device (no CPU path exists)")
        if not self._flat_is_intact():
            raise _L.EtpError("a parameter was re-allocated outside the flat buffer; call module._apply/.to() again")
        _L.require_device()
        _declare()
        _L.cast_bf16(self._flat, self._flat_bf16)
        self._cache_key = self._version_key()
        self._bf16_fresh = False
        if self._structs is None:
            self._structs = self._build_structs(self._flat.data_ptr(), self._flat_bf16.data_ptr(), 2)
        if self.precision == "high":
            self._refresh_hp(self._cache_key)

    # ------------------------------------------------------------------ high-precision inference mode
    def set_precision(self, precision: str):
        """``"bf16"`` (default): bf16 GEMM / attention operands, fp32 everywhere else — training and fast inference.
        ``"high"``: inference only; every GEMM is a split-bf16 x3 product on the tensor cores (fp32-class accuracy, 3x
        the GEMM work), attention in fp32: meets the reference's fp32 eval path (ss_trainer_ETP.py:513-756) within
        rtol 1e-3 / atol 1e-4 (tests/test_precision_gpu.py)."""
        if precision not in ("bf16", "high"):
            raise ValueError("precision must be 'bf16' or 'high'")
        self.precision = precision
        return self

    def _gemm_weight_names(self):
        # every 2-D parameter consumed as a GEMM B operand; the embedding TABLES (word / position / token-type / step /
        # nav-type: ``<...>embedding(s).weight``) are gathered in fp32 and skipped
        return [n for n, (_, _, shape) in self.layout.entries.items()
                if len(shape) == 2 and shape[1] % 64 == 0 and "embedding" not in n.split(".")[-2]]

    def _refresh_hp(self, key):
        """hi|hi|lo image of every GEMM weight ([out, 3*in] bf16 at element offset 3*off of ``_flat_hp``)."""
        if self._flat_hp is not None and self._hp_key == key and not self._bf16_fresh:
            return
        L = _L.lib()
        if self._flat_hp is None or self._flat_hp.device != self._flat.device:
            self._flat_hp = torch.zeros(3 * self.layout.total, dtype=torch.bfloat16, device=self._flat.device)
            self._structs_hp = None
        for n in self._gemm_weight_names():
            off, _, shape = self.layout.entries[n]
            _L._check(L.etp_split3(C.c_void_p(self._flat.data_ptr() + 4 * off), C.c_void_p(self._flat_hp.data_ptr() + 6 * off),
                                   shape[0], shape[1], 1, _L.stream_ptr()), "etp_split3")
        if self._structs_hp is None:
            self._structs_hp = self._build_structs(self._flat.data_ptr(), self._flat_hp.data_ptr(), 6)
            self._b32, self._b16, self._s16 = self._flat.data_ptr(), self._flat_bf16.data_ptr(), 2
        self._hp_key = key
        self._bf16_fresh = False

    def _hp_guard(self, wants_grad):
        if wants_grad:
            raise _L.EtpError("precision='high' is an inference mode (no backward exists for it): call under "
                              "torch.no_grad(), or set_precision('bf16') for training")

    # ------------------------------------------------------------------ ctypes weight structs
    def _version_key(self):
        return tuple(p._version for p in self._pmap.values())

    def _w32(self, name):
        return C.c_void_p(self._b32 + 4 * self.layout.offset(name))

    def _w16(self, name):
        return C.c_void_p(self._b16 + self._s16 * self.layout.offset(name))

    def _layer_struct(self, att, out, inter, outp, cross=None):
        lw = LayerWeights()
        if cross is not None:
            lw.xq_w, lw.xq_b = self._w16(cross + "att.query.weight"), self._w32(cross + "att.query.bias")
            lw.xkv_w, lw.xkv_b = self._w16(cross + "att.key.weight"), self._w32(cross + "att.key.bias")
            assert (self.layout.offset(cross + "att.value.weight")
                    == self.layout.offset(cross + "att.key.weight") + 768 * 768)
            lw.xo_w, lw.xo_b = self._w16(cross + "output.dense.weight"), self._w32(cross + "output.dense.bias")
            lw.xln_g, lw.xln_b = self._w32(cross + "output.LayerNorm.weight"), self._w32(cross + "output.LayerNorm.bias")
        lw.sqkv_w, lw.sqkv_b = self._w16(att + "query.weight"), self._w32(att + "query.bias")
        assert self.layout.offset(att + "value.weight") == self.layout.offset(att + "query.weight") + 2 * 768 * 768
        assert self.layout.offset(att + "value.bias") == self.layout.offset(att + "query.bias") + 2 * 768
        lw.so_w, lw.so_b = self._w16(out + "dense.weight"), self._w32(out + "dense.bias")
        lw.sln_g, lw.sln_b = self._w32(out + "LayerNorm.weight"), self._w32(out + "LayerNorm.bias")
        lw.f1_w, lw.f1_b = self._w16(inter + "dense.weight"), self._w32(inter + "dense.bias")
        lw.f2_w, lw.f2_b = self._w16(outp + "dense.weight"), self._w32(outp + "dense.bias")
        lw.fln_g, lw.fln_b = self._w32(outp + "LayerNorm.weight"), self._w32(outp + "LayerNorm.bias")
        return lw

    def _build_structs(self, b32, b16, s16):
        """ctypes structs over a flat buffer: b32 = base address of the fp32 image, b16/s16 = base address and
        element size of the image the GEMM-weight pointers refer to (bf16 parameters, or fp32 gradients)."""
        self._b32, self._b16, self._s16 = b32, b16, s16
        cfg = self.config
        s = {}
        X = cfg.num_x_layers
        xl = (LayerWeights * max(X, 1))()
        for i in range(X):
            p = f"global_encoder.encoder.x_layers.{i}."
            xl[i] = self._layer_struct(p + "visn_self_att.self.", p + "visn_self_att.output.", p + "visn_inter.",
                                       p + "visn_output.", cross=p + "visual_attention.")
        nw = NavWeights()
        nw.num_x_layers, nw.ln_eps, nw.layers = X, cfg.layer_norm_eps, xl
        nw.pos_w = self._w32("global_encoder.gmap_pos_embeddings.0.weight")
        nw.pos_b = self._w32("global_encoder.gmap_pos_embeddings.0.bias")
        nw.pos_g = self._w32("global_encoder.gmap_pos_embeddings.1.weight")
        nw.pos_bb = self._w32("global_encoder.gmap_pos_embeddings.1.bias")
        nw.step_emb = self._w32("global_encoder.gmap_step_embeddings.weight")
        if cfg.graph_sprels:
            nw.sprel_w = self._w32("global_encoder.sprel_linear.weight")
            nw.sprel_b = self._w32("global_encoder.sprel_linear.bias")
        nw.sap0_w, nw.sap0_b = self._w16("global_sap_head.net.0.weight"), self._w32("global_sap_head.net.0.bias")
        nw.sap_g, nw.sap_bb = self._w32("global_sap_head.net.2.weight"), self._w32("global_sap_head.net.2.bias")
        nw.sap4_w, nw.sap4_b = self._w32("global_sap_head.net.4.weight"), self._w32("global_sap_head.net.4.bias")
        if X > 0:
            k0 = "global_encoder.encoder.x_layers.0.visual_attention.att.key."
            nw.xkv_all_w, nw.xkv_all_b = self._w16(k0 + "weight"), self._w32(k0 + "bias")
            for i in range(X):  # [X*1536, 768] stacked key|value weights, [X*1536] biases
                ki = f"global_encoder.encoder.x_layers.{i}.visual_attention.att.key."
                assert self.layout.offset(ki + "weight") == self.layout.offset(k0 + "weight") + i * 2 * 768 * 768
                assert self.layout.offset(ki + "bias") == self.layout.offset(k0 + "bias") + i * 2 * 768
        s["nav"], s["nav_layers"] = nw, xl

        P = cfg.num_pano_layers
        pl = (PanoLayerWeights * max(P, 1))()
        for i in range(P):
            p = f"img_embeddings.pano_encoder.layers.{i}."
            w = PanoLayerWeights()
            w.in_w, w.in_b = self._w16(p + "self_attn.in_proj_weight"), self._w32(p + "self_attn.in_proj_bias")
            w.out_w, w.out_b = self._w16(p + "self_attn.out_proj.weight"), self._w32(p + "self_attn.out_proj.bias")
            w.l1_w, w.l1_b = self._w16(p + "linear1.weight"), self._w32(p + "linear1.bias")
            w.l2_w, w.l2_b = self._w16(p + "linear2.weight"), self._w32(p + "linear2.bias")
            w.n1_g, w.n1_b = self._w32(p + "norm1.weight"), self._w32(p + "norm1.bias")
            w.n2_g, w.n2_b = self._w32(p + "norm2.weight"), self._w32(p + "norm2.bias")
            pl[i] = w
        pw = PanoWeights()
        pw.num_pano_layers, pw.layer_eps, pw.layers = P, cfg.pano_layer_norm_eps, pl
        e = "img_embeddings."
        pw.img_w, pw.img_b = self._w16(e + "img_linear.weight"), self._w32(e + "img_linear.bias")
        if cfg.use_depth_embedding:
            pw.dep_w, pw.dep_b = self._w16(e + "dep_linear.weight"), self._w32(e + "dep_linear.bias")
            pw.dep_g, pw.dep_bb = self._w32(e + "dep_layer_norm.weight"), self._w32(e + "dep_layer_norm.bias")
        pw.loc_w, pw.loc_b = self._w32(e + "loc_linear.weight"), self._w32(e + "loc_linear.bias")
        pw.img_g, pw.img_bb = self._w32(e + "img_layer_norm.weight"), self._w32(e + "img_layer_norm.bias")
        pw.loc_g, pw.loc_bb = self._w32(e + "loc_layer_norm.weight"), self._w32(e + "loc_layer_norm.bias")
        pw.out_g, pw.out_bb = self._w32(e + "layer_norm.weight"), self._w32(e + "layer_norm.bias")
        pw.nav_emb = self._w32(e + "nav_type_embedding.weight")
        pw.tok_emb1 = C.c_void_p(self._w32("embeddings.token_type_embeddings.weight").value + 4 * 768)
        if P > 0:
            pw.fin_g, pw.fin_b = self._w32(e + "pano_encoder.norm.weight"), self._w32(e + "pano_encoder.norm.bias")
        s["pano"], s["pano_layers"] = pw, pl

        NL = cfg.num_l_layers
        tl = (LayerWeights * max(NL, 1))()
        for i in range(NL):
            p = f"lang_encoder.layer.{i}."
            tl[i] = self._layer_struct(p + "attention.self.", p + "attention.output.", p + "intermediate.", p + "output.")
        tw = TxtWeights()
        tw.num_l_layers, tw.ln_eps, tw.layers = NL, cfg.layer_norm_eps, tl
        tw.word_emb = self._w32("embeddings.word_embeddings.weight")
        tw.pos_emb = self._w32("embeddings.position_embeddings.weight")
        tw.type_emb0 = self._w32("embeddings.token_type_embeddings.weight")
        tw.emb_g, tw.emb_b = self._w32("embeddings.LayerNorm.weight"), self._w32("embeddings.LayerNorm.bias")
        s["txt"], s["txt_layers"] = tw, tl
        return s

    # ------------------------------------------------------------------ gradient plumbing
    def _group_names(self, group):
        from .layout import ordered_names
        if not hasattr(self, "_gnames"):
            self._gnames = ordered_names(self.config)
        return self._gnames[group]

    def _grad_view(self, gbuf, gstart, name):
        off, numel, shape = self.layout.entries[name]
        return gbuf[off - gstart: off - gstart + numel].view(shape)

    def _grad_structs_for(self, gbuf, gstart):
        """Weight-shaped structs whose every pointer lands in ``gbuf`` (fp32), which holds the flat-layout slice
        starting at element ``gstart``."""
        key = (gbuf.data_ptr(), gstart)
        st = self._grad_structs.get(key)
        if st is None:
            base = gbuf.data_ptr() - 4 * gstart
            st = self._build_structs(base, base, 4)
            self._b32, self._b16, self._s16 = self._flat.data_ptr(), self._flat_bf16.data_ptr(), 2
            if len(self._grad_structs) > 8:
                self._grad_structs.clear()
            self._grad_structs[key] = st
        return st

    def _grad_target(self, group):
        """(buffer, first element, per-call?) the backward of ``group`` accumulates into."""
        gs, ge = self.layout.group_ranges[group]
        if self._direct_grad is not None:
            return self._direct_grad, 0, False
        return torch.zeros(ge - gs, dtype=torch.float32, device=self._flat.device), gs, True

    def _anchor_t(self):
        if self._anchor.device != self._flat.device:
            self._anchor = torch.zeros(1, device=self._flat.device, requires_grad=True)
        return self._anchor

    # ------------------------------------------------------------------ dropout (train() mode)
    def set_dropout_seed(self, seed: int):
        """Restart the dropout seed stream (default: torch.initial_seed()); call k of forward_* uses seed stream[k]."""
        self._drop_base = int(seed) & 0xFFFFFFFFFFFFFFFF
        self._drop_calls = 0

    def set_dropout(self, p: float):
        """What ``set_dropout(model, p)`` of the pre-training driver does to every ``nn.Dropout`` of the reference
        (pretrain_src/pretrain_src/utils/misc.py:19-25): hidden, attention-probability and prediction-head dropout all
        become ``p``.  (This module has no ``nn.Dropout`` children for that helper to find: the probabilities live in the
        config and reach the kernels through ``etp_dropout``.)"""
        cfg = self.config
        cfg.hidden_dropout_prob = cfg.attention_probs_dropout_prob = cfg.pred_head_dropout_prob = float(p)

    def _next_dropout(self):
        """``etp_dropout`` of the next forward call, or None in eval() mode (or when every probability is 0)."""
        cfg = self.config
        if not self.training or max(cfg.hidden_dropout_prob, cfg.attention_probs_dropout_prob, cfg.pred_head_dropout_prob) <= 0:
            return None
        if self._drop_base is None:
            self._drop_base = torch.initial_seed() & 0xFFFFFFFFFFFFFFFF
        seed = (self._drop_base + 0x9E3779B97F4A7C15 * (self._drop_calls + 1)) & 0xFFFFFFFFFFFFFFFF
        self._drop_calls += 1
        return Dropout(seed, cfg.hidden_dropout_prob, cfg.attention_probs_dropout_prob, cfg.pred_head_dropout_prob)

    # ------------------------------------------------------------------ the three reference methods
    @staticmethod
    def _mask_u8(m):
        m = m.contiguous()
        return m.view(torch.uint8) if m.dtype == torch.bool else m.to(torch.uint8)

    def _wants_grad(self, group, *tensors):
        if not torch.is_grad_enabled():
            return False
        if any(t is not None and torch.is_tensor(t) and t.requires_grad for t in tensors):
            return True
        return any(self._pmap[n].requires_grad for n in self._group_names(group))

    def forward_txt(self, txt_ids, txt_masks):
        """vilmodel_cmt.py:684-688.  txt_ids int64 [B,L], txt_masks bool [B,L] -> txt_embeds fp32 [B,L,768]."""
        self._refresh_cache()
        if txt_ids.shape[1] > self.config.max_position_embeddings:
            raise ValueError("sequence longer than max_position_embeddings")
        ids = txt_ids.contiguous().long()
        mk = self._mask_u8(txt_masks)
        if self.precision == "high":
            self._hp_guard(self._wants_grad("txt") and self.config.update_lang_bert)
            return _txt_forward_hp(self, ids, mk)
        drop = self._next_dropout()
        if self._wants_grad("txt") and self.config.update_lang_bert:
            params = [] if self._direct_grad is not None else [self._pmap[n] for n in self._group_names("txt")]
            return _TxtFn.apply(self, ids, mk, drop, self._anchor_t(), *params)
        return _txt_forward(self, ids, mk, 0, drop)[0]

    def forward_panorama(self, rgb_fts, dep_fts, loc_fts, nav_types, view_lens):
        """vilmodel_cmt.py:690-719 -> (pano_embeds fp32 [B,V,768], pano_masks bool [B,V])."""
        self._refresh_cache()
        nt, vl = nav_types.contiguous().long(), view_lens.contiguous().long()
        loc = _f32c(loc_fts)
        if self.precision == "high":
            self._hp_guard(self._wants_grad("pano", rgb_fts, dep_fts))
            out, masks = _pano_forward_hp(self, _f32c(rgb_fts), _f32c(dep_fts), loc, nt, vl)
            return out, masks.view(torch.bool)
        drop = self._next_dropout()
        if self._wants_grad("pano", rgb_fts, dep_fts):
            params = [] if self._direct_grad is not None else [self._pmap[n] for n in self._pano_param_names()]
            return _PanoFn.apply(self, rgb_fts, dep_fts, loc, nt, vl, drop, self._anchor_t(), *params)
        out, masks, _, _ = _pano_forward(self, _f32c(rgb_fts), _f32c(dep_fts), loc, nt, vl, 0, drop)
        return out, masks.view(torch.bool)

    def _pano_param_names(self):
        # forward_panorama also reads row 1 of the token-type table (vilmodel_cmt.py:709), which lives in the txt group
        return self._group_names("pano") + ["embeddings.token_type_embeddings.weight"]

    def forward_navigation(self, txt_embeds, txt_masks, gmap_vpids, gmap_step_ids, gmap_img_fts, gmap_pos_fts,
                           gmap_masks, gmap_visited_masks, gmap_pair_dists):
        """vilmodel_cmt.py:721-750 -> {'gmap_embeds': fp32 [B,N,768], 'global_logits': fp32 [B,N]}.
        ``gmap_vpids`` is accepted and ignored, as in the reference."""
        self._refresh_cache()
        aux = (self._mask_u8(txt_masks), gmap_step_ids.contiguous().long(), _f32c(gmap_pos_fts),
               self._mask_u8(gmap_masks), self._mask_u8(gmap_visited_masks), _f32c(gmap_pair_dists))
        if isinstance(txt_embeds, TextKV):
            kv = txt_embeds
            if kv.grad is not None and kv.grad.done:
                raise _L.EtpError("this TextKV handle's backward has run: encode the instruction again for a new rollout")
            train = kv.grad is not None and torch.is_grad_enabled()
            if self.precision != "bf16" or (not train and self._wants_grad("nav", gmap_img_fts)):
                raise _L.EtpError("a TextKV handle serves the bf16 mode, and only one made by encode_text_kv with gradients "
                                  "enabled can be trained through")
            if len(kv) != gmap_img_fts.shape[0] or kv.length != txt_masks.shape[1]:
                raise ValueError("TextKV handle and the step's batch disagree: index the handle like all_txt_embeds")
            if train:
                drop = self._next_dropout()
                params = [] if self._direct_grad is not None else [self._pmap[n] for n in self._nav_kv_step_names()]
                embeds, logits = _NavKVFn.apply(self, kv.token, gmap_img_fts, kv, aux, drop, self._anchor_t(), *params)
            else:
                embeds, logits, _, _ = _nav_forward(self, kv, _f32c(gmap_img_fts), aux, 0, None)
            return {"gmap_embeds": embeds, "global_logits": logits}
        if self.precision == "high":
            self._hp_guard(self._wants_grad("nav", txt_embeds, gmap_img_fts))
            embeds, logits = _nav_forward_hp(self, _f32c(txt_embeds), _f32c(gmap_img_fts), aux)
            return {"gmap_embeds": embeds, "global_logits": logits}
        drop = self._next_dropout()
        if self._wants_grad("nav", txt_embeds, gmap_img_fts):
            params = [] if self._direct_grad is not None else [self._pmap[n] for n in self._group_names("nav")]
            embeds, logits = _NavFn.apply(self, txt_embeds, gmap_img_fts, aux, drop, self._anchor_t(), *params)
        else:
            embeds, logits, _, _ = _nav_forward(self, _txtc(txt_embeds), _f32c(gmap_img_fts), aux, 0, drop)
        return {"gmap_embeds": embeds, "global_logits": logits}

    def encode_text_kv(self, txt_embeds):
        """Once per episode (after ``forward_txt``): the key|value projections of the instruction for every x-layer, as a
        ``TextKV`` handle that ``forward_navigation`` accepts in place of ``txt_embeds``.
        Bit-identical to what the un-cached step computes; saves the [B*L,768] x [X*1536,768] GEMM at every step.

        With gradients enabled (bf16 mode, and ``txt_embeds`` or a cross-modal key/value weight requires grad) the handle
        can be trained through over a whole rollout: each step's backward adds its dK|dV into the handle's accumulator
        instead of running the text-side weight and data gradient GEMMs and keeping the step's K|V, and one node after the
        rollout runs them once.  Under ``torch.no_grad()`` it is an inference handle."""
        self._refresh_cache()
        X = self.config.num_x_layers
        if X == 0:
            raise ValueError("no cross-modal layers: nothing to cache")
        if torch.is_grad_enabled() and self.precision == "bf16" and (
                txt_embeds.requires_grad or any(self._pmap[n].requires_grad for n in self._kv_weight_names())):
            params = [] if self._direct_grad is not None else [self._pmap[n] for n in self._kv_weight_names()]
            box = []
            token = _TextKVFn.apply(self, txt_embeds, box, self._anchor_t(), *params)
            kv, grad = box
            return TextKV(kv, txt_embeds.shape[0], txt_embeds.shape[1], grad=grad, token=token)
        t = _txtc(txt_embeds)
        return TextKV(_encode_text_kv(self, t), t.shape[0], t.shape[1])

    def _kv_weight_names(self):
        # key|value weights of every cross-modal layer: the stacked [X*1536, 768] operand of the text K|V GEMM
        return [f"global_encoder.encoder.x_layers.{i}.visual_attention.att.{kv}.weight"
                for i in range(self.config.num_x_layers) for kv in ("key", "value")]

    def _nav_kv_step_names(self):
        # the navigation group minus the key|value weights, whose gradient the training TextKV handle's node returns
        kvw = set(self._kv_weight_names())
        return [n for n in self._group_names("nav") if n not in kvw]

    # ------------------------------------------------------------------ training helper
    def make_trainer(self, lr=1e-5, world_size=1, **kw):
        return PlannerTrainer(self, lr=lr, world_size=world_size, **kw)


# ----------------------------------------------------------------------------------------------------
# raw step calls (no autograd)
# ----------------------------------------------------------------------------------------------------
def _dptr(drop):
    return C.byref(drop) if drop is not None else None


def _txt_forward(m, ids, mk, training, drop=None):
    B, Lt = ids.shape
    L = _L.lib()
    out = torch.empty(B, Lt, 768, device=ids.device, dtype=torch.float32)
    nbytes = L.etp_txt_saved_bytes(B, Lt, m.config.num_l_layers, training)
    saved = torch.empty(nbytes, dtype=torch.uint8, device=ids.device)
    _L._check(L.etp_forward_txt(C.byref(m._structs["txt"]), _L.ptr(ids), _L.ptr(mk), B, Lt, _L.ptr(out), _L.ptr(saved),
                                nbytes, training, _L.stream_ptr(), _dptr(drop)), "etp_forward_txt")
    return out, saved


def _pano_inputs(rgb, dep, loc, nt, vl, drop=None):
    pi = PanoInputs()
    if drop is not None:
        pi.dropout = C.pointer(drop)
    pi.B, pi.V = rgb.shape[0], rgb.shape[1]
    pi.rgb_fts, pi.dep_fts, pi.loc_fts = _L.ptr(rgb), _L.ptr(dep), _L.ptr(loc)
    pi.nav_types, pi.view_lens = _L.ptr(nt), _L.ptr(vl)
    return pi


def _pano_forward(m, rgb, dep, loc, nt, vl, training, drop=None):
    B, V = rgb.shape[:2]
    L = _L.lib()
    out = torch.empty(B, V, 768, device=rgb.device, dtype=torch.float32)
    masks = torch.empty(B, V, device=rgb.device, dtype=torch.uint8)
    pi = _pano_inputs(rgb, dep, loc, nt, vl, drop)
    nbytes = L.etp_pano_saved_bytes(B, V, m.config.num_pano_layers, training)
    saved = torch.empty(nbytes, dtype=torch.uint8, device=rgb.device)
    _L._check(L.etp_forward_panorama(C.byref(m._structs["pano"]), C.byref(pi), _L.ptr(out), _L.ptr(masks), _L.ptr(saved),
                                     nbytes, training, _L.stream_ptr()), "etp_forward_panorama")
    return out, masks, saved, pi


def _nav_inputs(txt, img, aux, drop=None):
    tm, ids, pos, gm, vm, pd = aux
    ni = NavInputs()
    if drop is not None:
        ni.dropout = C.pointer(drop)
    ni.B, ni.N, ni.L = img.shape[0], img.shape[1], txt.shape[1]
    if isinstance(txt, TextKV):         # episode-level K|V cache (+ the surviving episodes' row map)
        ni.txt_kv_all, ni.txt_kv_batch = _L.ptr(txt.kv_all), txt.batch
        ni.txt_kv_rows = _L.ptr(txt.rows)
        ni._keep = txt
    elif txt.dtype == torch.bfloat16:   # bf16 instruction embeddings are consumed as they are (etp_nav_inputs.txt_embeds_bf16)
        ni.txt_embeds_bf16 = _L.ptr(txt)
    else:
        ni.txt_embeds = _L.ptr(txt)
    ni.txt_masks, ni.gmap_step_ids = _L.ptr(tm), _L.ptr(ids)
    ni.gmap_img_fts, ni.gmap_pos_fts, ni.gmap_masks = _L.ptr(img), _L.ptr(pos), _L.ptr(gm)
    ni.gmap_visited_masks, ni.gmap_pair_dists = _L.ptr(vm), _L.ptr(pd)
    return ni


def _encode_text_kv(m, t):
    """etp_encode_text_kv of txt_embeds ``t`` (fp32 or bf16 [B,L,768]) -> bf16 [B*L, X*1536]."""
    B, Lt = t.shape[:2]
    kv = torch.empty(B * Lt, m.config.num_x_layers * 1536, dtype=torch.bfloat16, device=t.device)
    work = torch.empty(B * Lt * 768, dtype=torch.bfloat16, device=t.device) if t.dtype != torch.bfloat16 else None
    _L._check(_L.lib().etp_encode_text_kv(C.byref(m._structs["nav"]), _L.ptr(t) if work is not None else None,
                                          _L.ptr(t) if work is None else None, B, Lt, _L.ptr(kv), _L.ptr(work),
                                          _L.stream_ptr()), "etp_encode_text_kv")
    return kv


def _nav_forward(m, txt, img, aux, training, drop=None, img_ready_event=None, side_sm_reserve=0):
    B, N = img.shape[:2]
    Lt = txt.shape[1]
    L = _L.lib()
    ni = _nav_inputs(txt, img, aux, drop)
    if img_ready_event is not None:
        ni.img_ready_event = C.c_void_p(img_ready_event)
    ni.side_sm_reserve = side_sm_reserve
    embeds = torch.empty(B, N, 768, device=img.device, dtype=torch.float32)
    logits = torch.empty(B, N, device=img.device, dtype=torch.float32)
    saved_bytes = L.etp_nav_kv_saved_bytes if isinstance(txt, TextKV) else L.etp_nav_saved_bytes
    nbytes = saved_bytes(B, N, Lt, m.config.num_x_layers, training)
    saved = torch.empty(nbytes, dtype=torch.uint8, device=img.device)
    _L._check(L.etp_forward_navigation(C.byref(m._structs["nav"]), C.byref(ni), _L.ptr(embeds), _L.ptr(logits),
                                       _L.ptr(saved), nbytes, training, _L.stream_ptr()), "etp_forward_navigation")
    return embeds, logits, saved, ni


def _txt_forward_hp(m, ids, mk):
    B, Lt = ids.shape
    L = _L.lib()
    out = torch.empty(B, Lt, 768, device=ids.device, dtype=torch.float32)
    nbytes = L.etp_hp_txt_work_bytes(B, Lt)
    work = torch.empty(nbytes, dtype=torch.uint8, device=ids.device)
    _L._check(L.etp_forward_txt_hp(C.byref(m._structs_hp["txt"]), _L.ptr(ids), _L.ptr(mk), B, Lt, _L.ptr(out), _L.ptr(work),
                                   nbytes, _L.stream_ptr()), "etp_forward_txt_hp")
    return out


def _pano_forward_hp(m, rgb, dep, loc, nt, vl):
    B, V = rgb.shape[:2]
    L = _L.lib()
    out = torch.empty(B, V, 768, device=rgb.device, dtype=torch.float32)
    masks = torch.empty(B, V, device=rgb.device, dtype=torch.uint8)
    pi = _pano_inputs(rgb, dep, loc, nt, vl)
    nbytes = L.etp_hp_pano_work_bytes(B, V)
    work = torch.empty(nbytes, dtype=torch.uint8, device=rgb.device)
    _L._check(L.etp_forward_panorama_hp(C.byref(m._structs_hp["pano"]), C.byref(pi), _L.ptr(out), _L.ptr(masks), _L.ptr(work),
                                        nbytes, _L.stream_ptr()), "etp_forward_panorama_hp")
    return out, masks


def _nav_forward_hp(m, txt, img, aux):
    B, N = img.shape[:2]
    Lt = txt.shape[1]
    L = _L.lib()
    ni = _nav_inputs(txt, img, aux)
    embeds = torch.empty(B, N, 768, device=img.device, dtype=torch.float32)
    logits = torch.empty(B, N, device=img.device, dtype=torch.float32)
    nbytes = L.etp_hp_nav_work_bytes(B, N, Lt, m.config.num_x_layers)
    work = torch.empty(nbytes, dtype=torch.uint8, device=img.device)
    _L._check(L.etp_forward_navigation_hp(C.byref(m._structs_hp["nav"]), C.byref(ni), _L.ptr(embeds), _L.ptr(logits),
                                          _L.ptr(work), nbytes, _L.stream_ptr()), "etp_forward_navigation_hp")
    return embeds, logits


def _nav_backward_raw(m, txt, img, aux, drop, saved, de, dl, want_dtxt, want_dimg, img_grad_event=None, side_sm_reserve=0,
                      d_img_out=None):
    """etp_backward_navigation on the current stream; parameter gradients go to m._grad_target('nav').
    Returns (d_txt, d_img, gbuf, gstart, per_call)."""
    L = _L.lib()
    B, N, Lt = img.shape[0], img.shape[1], txt.shape[1]
    gbuf, gstart, per_call = m._grad_target("nav")
    gst = m._grad_structs_for(gbuf, gstart)
    ni = _nav_inputs(txt, img, aux, drop)
    if m._layer_events is not None:
        ni.layer_done_events = m._layer_events
    if img_grad_event is not None:
        ni.img_grad_event = C.c_void_p(img_grad_event)
    ni.side_sm_reserve = side_sm_reserve
    if isinstance(txt, TextKV):
        ni.txt_kv_grad = _L.ptr(txt.grad.acc)
    d_txt = torch.empty(txt.shape, dtype=torch.float32, device=img.device) if want_dtxt else None
    d_img = (d_img_out if d_img_out is not None else torch.empty_like(img)) if want_dimg else None
    wbytes = L.etp_nav_bwd_work_bytes(B, N, Lt, m.config.num_x_layers)
    work = torch.empty(wbytes, dtype=torch.uint8, device=img.device)
    _L._check(L.etp_backward_navigation(C.byref(m._structs["nav"]), C.byref(gst["nav"]), C.byref(ni), _L.ptr(de),
                                        _L.ptr(dl), _L.ptr(saved), saved.numel(), _L.ptr(work), wbytes,
                                        _L.ptr(d_txt), _L.ptr(d_img), _L.stream_ptr()), "etp_backward_navigation")
    return d_txt, d_img, gbuf, gstart, per_call


def _pano_backward_raw(m, rgb, dep, loc, nt, vl, masks, drop, saved, d_out, want_drgb, want_ddep):
    """etp_backward_panorama on the current stream.  Returns (d_rgb, d_dep, gbuf, gstart, per_call, tok) where ``tok`` is
    the per-call token-type row-1 gradient (None in the trainer's direct-gradient mode)."""
    L = _L.lib()
    B, V = rgb.shape[:2]
    gs, ge = m.layout.group_ranges["pano"]
    if m._direct_grad is not None:
        gbuf, gstart, per_call = m._direct_grad, 0, False
        gst = m._grad_structs_for(gbuf, gstart)
        tok = None
        if getattr(m, "_tok_scratch", None) is not None:
            gst["pano"].tok_emb1 = C.c_void_p(m._tok_scratch.data_ptr())
    else:
        # group-sized scratch + 768 extra floats for the token-type row 1, which lives in the txt group
        gbuf = torch.zeros(ge - gs + 768, dtype=torch.float32, device=rgb.device)
        gstart, per_call = gs, True
        gst = m._grad_structs_for(gbuf, gstart)
        tok = gbuf[ge - gs:]
        gst["pano"].tok_emb1 = C.c_void_p(tok.data_ptr())
    pi = _pano_inputs(rgb, dep, loc, nt, vl, drop)
    if getattr(m, "_pano_layer_events", None) is not None:
        pi.layer_done_events = m._pano_layer_events
    d_rgb = torch.empty_like(rgb) if want_drgb else None
    d_dep = torch.empty_like(dep) if (want_ddep and m.config.use_depth_embedding) else None
    wbytes = L.etp_pano_bwd_work_bytes(B, V)
    work = torch.empty(wbytes, dtype=torch.uint8, device=rgb.device)
    _L._check(L.etp_backward_panorama(C.byref(m._structs["pano"]), C.byref(gst["pano"]), C.byref(pi), _L.ptr(masks),
                                      _L.ptr(_f32c(d_out)), _L.ptr(saved), saved.numel(), _L.ptr(work), wbytes,
                                      _L.ptr(d_rgb), _L.ptr(d_dep), _L.stream_ptr()), "etp_backward_panorama")
    return d_rgb, d_dep, gbuf, gstart, per_call, tok


# ----------------------------------------------------------------------------------------------------
# autograd glue: one node per reference method; backward = one step-level C call
# ----------------------------------------------------------------------------------------------------
def _param_grads(m, names, gbuf, gstart, per_call, nparams):
    if nparams == 0 or not per_call:
        return [None] * nparams
    return [m._grad_view(gbuf, gstart, n) if m._pmap[n].requires_grad else None for n in names]


class _NavFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, m, txt_embeds, gmap_img_fts, aux, drop, anchor, *params):
        txt, img = _txtc(txt_embeds), _f32c(gmap_img_fts)
        embeds, logits, saved, _ = _nav_forward(m, txt, img, aux, 1, drop)
        ctx.m, ctx.saved, ctx.keep, ctx.nparams, ctx.drop = m, saved, (txt, img, aux), len(params), drop
        ctx.in_dtypes = (txt_embeds.dtype, gmap_img_fts.dtype)
        return embeds, logits

    @staticmethod
    def backward(ctx, d_embeds, d_logits):
        m = ctx.m
        txt, img, aux = ctx.keep
        de = _f32c(d_embeds) if d_embeds is not None else None
        dl = _f32c(d_logits) if d_logits is not None else None
        if dl is not None:
            dl = torch.nan_to_num(dl, nan=0.0, posinf=0.0, neginf=0.0)
        d_txt, d_img, gbuf, gstart, per_call = _nav_backward_raw(m, txt, img, aux, ctx.drop, ctx.saved, de, dl,
                                                                 ctx.needs_input_grad[1], ctx.needs_input_grad[2])
        pg = _param_grads(m, m._group_names("nav"), gbuf, gstart, per_call, ctx.nparams)
        if d_txt is not None and d_txt.dtype != ctx.in_dtypes[0]:
            d_txt = d_txt.to(ctx.in_dtypes[0])
        if d_img is not None and d_img.dtype != ctx.in_dtypes[1]:
            d_img = d_img.to(ctx.in_dtypes[1])
        return (None, d_txt, d_img, None, None, None, *pg)


class _TextKVFn(torch.autograd.Function):
    """encode_text_kv of a training rollout.  Output: a token the navigation steps that read the handle take as input, so
    that this node's backward runs after all of theirs; it turns the accumulated dK|dV into the key|value weight gradient
    and d txt_embeds (one GEMM each)."""

    @staticmethod
    def forward(ctx, m, txt_embeds, box, anchor, *params):
        t = _txtc(txt_embeds)
        kv = _encode_text_kv(m, t)
        grad = _TextKVGrad(torch.zeros(kv.shape, dtype=torch.float32, device=kv.device))
        box.extend((kv, grad))
        ctx.m, ctx.t, ctx.grad, ctx.nparams, ctx.in_dtype = m, t, grad, len(params), txt_embeds.dtype
        return torch.zeros(1, device=kv.device)

    @staticmethod
    def backward(ctx, _d_token):
        m, t, grad = ctx.m, ctx.t, ctx.grad
        if grad.done:
            raise _L.EtpError("the TextKV handle's backward already ran (retain_graph is not supported through it)")
        L = _L.lib()
        B, Lt = t.shape[:2]
        gbuf, gstart, per_call = m._grad_target("nav")
        gst = m._grad_structs_for(gbuf, gstart)
        d_txt = torch.empty(t.shape, dtype=torch.float32, device=t.device) if ctx.needs_input_grad[1] else None
        work = torch.empty(L.etp_text_kv_bwd_work_bytes(B, Lt, m.config.num_x_layers), dtype=torch.uint8, device=t.device)
        bf = t.dtype == torch.bfloat16
        _L._check(L.etp_backward_text_kv(C.byref(m._structs["nav"]), C.byref(gst["nav"]), None if bf else _L.ptr(t),
                                         _L.ptr(t) if bf else None, B, Lt, _L.ptr(grad.acc), _L.ptr(d_txt), _L.ptr(work),
                                         _L.stream_ptr()), "etp_backward_text_kv")
        grad.done, grad.acc = True, None
        pg = _param_grads(m, m._kv_weight_names(), gbuf, gstart, per_call, ctx.nparams)
        if d_txt is not None and d_txt.dtype != ctx.in_dtype:
            d_txt = d_txt.to(ctx.in_dtype)
        return (None, d_txt, None, None, *pg)


class _NavKVFn(torch.autograd.Function):
    """forward_navigation through a training TextKV handle: the record leaves out the step's K|V and bf16 txt_embeds, and
    the backward adds dK|dV into the handle's accumulator (the token's gradient is zero)."""

    @staticmethod
    def forward(ctx, m, token, gmap_img_fts, kv, aux, drop, anchor, *params):
        img = _f32c(gmap_img_fts)
        embeds, logits, saved, _ = _nav_forward(m, kv, img, aux, 1, drop)
        # the handle minus its token: the token's node must not be kept alive from here
        ctx.kv = TextKV(kv.kv_all, kv.batch, kv.length, kv.rows, kv.grad)
        ctx.m, ctx.saved, ctx.keep, ctx.nparams, ctx.drop = m, saved, (img, aux), len(params), drop
        ctx.in_dtype = gmap_img_fts.dtype
        return embeds, logits

    @staticmethod
    def backward(ctx, d_embeds, d_logits):
        m, kv = ctx.m, ctx.kv
        img, aux = ctx.keep
        if kv.grad.done:
            raise _L.EtpError("the TextKV handle's backward already ran (retain_graph is not supported through it)")
        de = _f32c(d_embeds) if d_embeds is not None else None
        dl = _f32c(d_logits) if d_logits is not None else None
        if dl is not None:
            dl = torch.nan_to_num(dl, nan=0.0, posinf=0.0, neginf=0.0)
        _, d_img, gbuf, gstart, per_call = _nav_backward_raw(m, kv, img, aux, ctx.drop, ctx.saved, de, dl, False,
                                                             ctx.needs_input_grad[2])
        pg = _param_grads(m, m._nav_kv_step_names(), gbuf, gstart, per_call, ctx.nparams)
        if d_img is not None and d_img.dtype != ctx.in_dtype:
            d_img = d_img.to(ctx.in_dtype)
        d_token = torch.zeros(1, device=img.device) if ctx.needs_input_grad[1] else None
        return (None, d_token, d_img, None, None, None, None, *pg)


class _PanoFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, m, rgb_fts, dep_fts, loc, nt, vl, drop, anchor, *params):
        rgb, dep = _f32c(rgb_fts), _f32c(dep_fts)
        out, masks, saved, _ = _pano_forward(m, rgb, dep, loc, nt, vl, 1, drop)
        ctx.m, ctx.saved, ctx.keep, ctx.nparams, ctx.drop = m, saved, (rgb, dep, loc, nt, vl, masks), len(params), drop
        ctx.in_dtypes = (rgb_fts.dtype, dep_fts.dtype)
        mb = masks.view(torch.bool)
        ctx.mark_non_differentiable(mb)
        return out, mb

    @staticmethod
    def backward(ctx, d_out, _unused):
        m = ctx.m
        rgb, dep, loc, nt, vl, masks = ctx.keep
        d_rgb, d_dep, gbuf, gstart, per_call, tok = _pano_backward_raw(m, rgb, dep, loc, nt, vl, masks, ctx.drop, ctx.saved, d_out,
                                                                       ctx.needs_input_grad[1], ctx.needs_input_grad[2])
        pg = []
        if ctx.nparams:
            names = m._pano_param_names()
            pg = _param_grads(m, names[:-1], gbuf, gstart, per_call, ctx.nparams - 1)
            tt = None
            if per_call and m._pmap[names[-1]].requires_grad:
                tt = torch.zeros_like(m._pmap[names[-1]])
                tt[1] = tok
            pg.append(tt)
        if d_dep is None and ctx.needs_input_grad[2]:
            d_dep = torch.zeros_like(dep)
        if d_rgb is not None and d_rgb.dtype != ctx.in_dtypes[0]:
            d_rgb = d_rgb.to(ctx.in_dtypes[0])
        if d_dep is not None and d_dep.dtype != ctx.in_dtypes[1]:
            d_dep = d_dep.to(ctx.in_dtypes[1])
        return (None, d_rgb, d_dep, None, None, None, None, None, *pg)


class _TxtFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, m, ids, mk, drop, anchor, *params):
        out, saved = _txt_forward(m, ids, mk, 1, drop)
        ctx.m, ctx.saved, ctx.keep, ctx.nparams, ctx.drop = m, saved, (ids, mk), len(params), drop
        return out

    @staticmethod
    def backward(ctx, d_out):
        m = ctx.m
        ids, mk = ctx.keep
        L = _L.lib()
        B, Lt = ids.shape
        gbuf, gstart, per_call = m._grad_target("txt")
        gst = m._grad_structs_for(gbuf, gstart)
        wbytes = L.etp_txt_bwd_work_bytes(B, Lt)
        work = torch.empty(wbytes, dtype=torch.uint8, device=ids.device)
        _L._check(L.etp_backward_txt(C.byref(m._structs["txt"]), C.byref(gst["txt"]), _L.ptr(ids), _L.ptr(mk), B, Lt,
                                     _L.ptr(_f32c(d_out)), _L.ptr(ctx.saved), ctx.saved.numel(), _L.ptr(work), wbytes,
                                     _L.stream_ptr(), _dptr(ctx.drop)), "etp_backward_txt")
        pg = _param_grads(m, m._group_names("txt"), gbuf, gstart, per_call, ctx.nparams)
        return (None, None, None, None, None, *pg)


class PeerGroup(C.Structure):
    """etp_peer_group (include/etpnav_b200.h): every rank's flat gradient / parameter / bf16-image / flag buffers."""
    _fields_ = [("world", i32), ("rank", i32), ("grad", p_void * 8), ("param", p_void * 8), ("image", p_void * 8),
                ("flags", p_void * 8)]


PEER_FLAG_WORDS = 2 * 32 * 8
# peer allocations this process has mapped: (peer rank, IPC handle) -> [base pointer, users].  Two trainers of one process
# can see the same peer allocation (small tensors share an allocator segment); a handle is opened once and closed with
# its last user.
_IPC_OPEN = {}


def _ipc_open(rank, handle):
    ent = _IPC_OPEN.get((rank, handle))
    if ent is None:
        base = p_void()
        _L._check(_L.lib().etp_ipc_open(handle, C.byref(base)), "etp_ipc_open")
        ent = _IPC_OPEN[(rank, handle)] = [base.value, 0]
    ent[1] += 1
    return ent[0]


def _ipc_release(rank, handle):
    ent = _IPC_OPEN.get((rank, handle))
    if ent is not None:
        ent[1] -= 1
        if ent[1] <= 0:
            del _IPC_OPEN[(rank, handle)]
            _L.lib().etp_ipc_close(C.c_void_p(ent[0]))


def peer_partition(x, y, world, rank):
    """Sub-slice of the trainable run [x, y) that `rank` owns in the peer-memory update: `world` equal chunks, rounded up
    to the 64-element granule of the flat layout; trailing ranks may own nothing."""
    chunk = (-(-(y - x) // world) + 63) // 64 * 64
    x0 = min(y, x + rank * chunk)
    return x0, min(y, x0 + chunk)


class PlannerTrainer:
    """Fused training step for the planner hot path: forward_panorama + forward_navigation, the caller-side loss of
    ss_trainer_ETP.py:890-892 (cross-entropy, sum over the batch, divided by the number of actions as :1055),
    backward through the step-level C calls accumulating straight into one flat fp32 gradient buffer, ONE NCCL
    all-reduce of that buffer's step slice (the reference's DDP mean, ss_trainer_ETP.py:211-212) and a fused
    AdamW (torch.optim.AdamW defaults, :213) that also refreshes the bf16 weight image."""

    def __init__(self, model, lr=1e-5, world_size=1, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2, groups=("pano", "nav"),
                 grad_comm="fp32", comm_sms=0, overlap=True, pano_sms=28):
        """``grad_comm``: dtype the gradient buckets cross NVLink in — "fp32" (DDP's default, the reference) or "bf16"
        (each bucket is rounded to bf16 for the all-reduce and widened again: half the bytes, like DDP's bf16 compression
        hook; gradients are still ACCUMULATED and applied in fp32).  ``comm_sms``: SMs the library's persistent grids leave
        to the collective's CTAs while training data-parallel (etp_set_sm_reserve; pair it with NCCL_MAX_CTAS)."""
        self.m, self.lr, self.world, self.betas, self.eps, self.wd = model, lr, world_size, betas, eps, weight_decay
        if grad_comm not in ("fp32", "bf16", "peer"):
            raise ValueError("grad_comm must be 'fp32', 'bf16' or 'peer'")
        if grad_comm == "peer" and world_size == 1:
            grad_comm = "fp32"
        self._peer, self._peer_plan, self._peer_bases, self.peer_fallback = None, None, [], None
        self._grads_clean, self._clear_after_update = False, False
        self._pipelined, self._pending_join, self._ev_nav, self._k_nav = False, False, None, -1
        self._debug_pano_start = None
        self.grad_comm, self.comm_sms, self._comm_buf = grad_comm, int(comm_sms), None
        # panorama branch on its own stream next to the instruction-side GEMMs of the navigation call
        # (_forward_backward_overlapped); ETP_OVERLAP=0 / overlap=False runs the two calls back to back through autograd
        import os as _os0
        self.overlap = bool(overlap) and _os0.environ.get("ETP_OVERLAP", "1") != "0"
        self.pano_sms = int(_os0.environ.get("ETP_PANO_SMS", pano_sms))
        self.pano_stream, self._ev_img, self._ev_dimg = None, None, None
        self._bufs, self._seen_inputs = {}, set()
        dev = model._flat.device
        if world_size > 1:
            # DDP broadcasts rank 0's parameters when it wraps the module (ss_trainer_ETP.py:211-212): replicas built from
            # different seeds, or loaded on one rank only, must not silently diverge while their gradients are averaged
            import torch.distributed as dist
            with torch.no_grad():
                dist.broadcast(model._flat, src=0)
            model._cache_key = None
            # ... and every rank must draw its own dropout masks
            if model._drop_base is None:
                model._drop_base = (torch.initial_seed() + 0x9E3779B97F4A7C15 * (dist.get_rank() + 1)) & 0xFFFFFFFFFFFFFFFF
        model._refresh_cache()
        model._direct_grad = torch.zeros(model.layout.total, dtype=torch.float32, device=dev)
        self.lo = min(model.layout.group_ranges[g][0] for g in groups)
        self.hi = max(model.layout.group_ranges[g][1] for g in groups)
        n = self.hi - self.lo
        self.t = 0
        # torch.optim.AdamW skips parameters without a gradient (frozen by fix_pano_embedding / fix_lang_embedding,
        # vilmodel_cmt.py:675-682): only the runs of the slice whose parameters require a gradient are stepped (one run
        # when nothing is frozen), so frozen weights see neither an update nor weight decay
        self.active = self._active_ranges(model, self.lo, self.hi)
        # forward_panorama reads row 1 of the token-type table, which lives in the txt group: when that group is not
        # stepped here its gradient goes to a scratch row instead of piling up, unapplied, in the flat gradient buffer
        gs, ge = model.layout.group_ranges["txt"]
        model._tok_scratch = None if (self.lo <= gs and ge <= self.hi) else torch.zeros(768, dtype=torch.float32, device=dev)
        # The update runs bucket by bucket, in the order the backward completes the buckets, on a SIDE stream: x-layer i's
        # bucket starts as soon as the event the nav backward records for it fires, so its (data-parallel) all-reduce and
        # its AdamW run under the rest of the backward; only the last bucket (panorama group) is exposed.
        from .dist import gradient_buckets
        self.buckets = [(nm, a - self.lo, b - self.lo) for nm, a, b in
                        gradient_buckets(model.layout, model.config, self.lo, self.hi)]
        self.side, self._events = None, []
        # index of the last bucket of the navigation group (x-layers, then node packing / text K|V): the compute stream of a
        # pipelined step() only waits for the update up to here; the panorama buckets finish under the next step's start
        self._k_nav = max((i for i, (nm, _, _) in enumerate(self.buckets) if nm.startswith("x_layer_") or nm == "nav_head"),
                          default=-1)
        if dev.type == "cuda":
            self._ev_nav = torch.cuda.Event()
            self.side = torch.cuda.Stream(dev)
            self.pano_stream = torch.cuda.Stream(dev)
            _Le = _L.lib()
            _Le.etp_event_create.restype = p_void
            _Le.etp_event_record.argtypes = [p_void, p_void]
            _Le.etp_stream_wait_event.argtypes = [p_void, p_void]
            self._ev_img, self._ev_dimg = _Le.etp_event_create(), _Le.etp_event_create()
            L0 = _L.lib()
            L0.etp_event_create.restype = p_void
            L0.etp_event_destroy.argtypes = [p_void]
            L0.etp_stream_wait_event.argtypes = [p_void, p_void]
            X = model.config.num_x_layers
            self._events = [L0.etp_event_create() for _ in range(X + 1)]   # one per x-layer + "nav group complete"
            model._layer_events = (p_void * (X + 1))(*self._events)
            Pn = model.config.num_pano_layers
            self._pano_events = [None] + [L0.etp_event_create() for _ in range(1, Pn)]
            model._pano_layer_events = (p_void * max(Pn, 1))(*self._pano_events) if Pn > 1 else None
            # the update runs UNDER the backward: a small grid-striding grid, so it does not take the registers / thread
            # slots the persistent GEMM CTA pairs need (ETP_ADAMW_CTAS overrides: 16 = the stand-alone roofline grid)
            import os as _os
            L0.etp_set_adamw_ctas_per_sm.argtypes = [i32]
            L0.etp_set_adamw_ctas_per_sm(int(_os.environ.get("ETP_ADAMW_CTAS", "4")))
            if world_size > 1:
                L0.etp_set_sm_reserve.argtypes = [i32]
                L0.etp_set_sm_reserve(self.comm_sms)
                if self.grad_comm == "peer":
                    self._peer_setup()
                if self.grad_comm == "bf16":
                    self._comm_buf = torch.empty(n, dtype=torch.bfloat16, device=dev)
        elif self.grad_comm == "peer":
            raise RuntimeError("grad_comm='peer' needs CUDA devices (peer memory over NVLink)")
        if self._peer is None:
            self.exp_avg = torch.zeros(n, dtype=torch.float32, device=dev)
            self.exp_avg_sq = torch.zeros(n, dtype=torch.float32, device=dev)
        L = _L.lib()
        L.etp_adamw_step.argtypes = [p_void, p_void, p_void, p_void, p_void, C.c_int64, f32, f32, f32, f32, f32, i32, f32,
                                     p_void]

    # ---- data-parallel update over NVLink peer memory (csrc/peer.cu) -------------------------------------------------
    def _peer_setup(self):
        """Map every rank's flat gradient / parameter / bf16-image buffers and flag block (CUDA IPC), cut every bucket's
        trainable runs into per-rank sub-slices and allocate the optimizer state of the OWNED sub-slices only.  If any
        rank cannot export / map (IPC not permitted in this container, no peer access) all ranks fall back to the NCCL
        all-reduce path together; ``peer_fallback`` keeps the reason."""
        import torch.distributed as dist
        m, L0 = self.m, _L.lib()
        rank, world, dev = dist.get_rank(), self.world, m._flat.device
        L0.etp_ipc_export.argtypes = [p_void, p_void, C.POINTER(C.c_int64)]
        L0.etp_ipc_open.argtypes = [p_void, C.POINTER(p_void)]
        L0.etp_ipc_close.argtypes = [p_void]
        L0.etp_peer_signal.argtypes = [C.POINTER(PeerGroup), i32, i32, C.c_uint32, p_void]
        L0.etp_peer_wait.argtypes = [C.POINTER(PeerGroup), i32, i32, i32, C.c_uint32, C.c_double, p_void]
        L0.etp_peer_reduce_adamw.argtypes = [C.POINTER(PeerGroup), C.c_int64, C.c_int64, p_void, p_void, f32, f32, f32, f32,
                                             f32, i32, i32, i32, p_void]
        L0.etp_peer_error.argtypes = [C.POINTER(i32)]
        self._peer_flags = torch.zeros(PEER_FLAG_WORDS, dtype=torch.int32, device=dev)
        bufs = {"grad": m._direct_grad, "param": m._flat, "image": m._flat_bf16, "flags": self._peer_flags}
        torch.cuda.synchronize(dev)
        mine, why = {}, None
        try:
            if world > 8:
                raise RuntimeError("more than 8 ranks")
            for k, t in bufs.items():
                h, off = (C.c_ubyte * 64)(), C.c_int64()
                _L._check(L0.etp_ipc_export(C.c_void_p(t.data_ptr()), h, C.byref(off)), "etp_ipc_export")
                mine[k] = (bytes(h), off.value)
        except Exception as e:  # noqa: BLE001 - reported, and every rank takes the same fallback
            why = f"rank {rank}: {e}"
        allh = [None] * world
        dist.all_gather_object(allh, (mine, why))
        g = PeerGroup()
        g.world, g.rank = world, rank
        opened = {}
        if not any(w for _, w in allh):
            try:
                for r in range(world):
                    for k, t in bufs.items():
                        if r == rank:
                            ptr = t.data_ptr()
                        else:
                            hb, off = allh[r][0][k]
                            if (r, hb) not in opened:
                                opened[(r, hb)] = _ipc_open(r, hb)
                            ptr = opened[(r, hb)] + off
                        getattr(g, k)[r] = ptr
            except Exception as e:  # noqa: BLE001
                why = f"rank {rank}: {e}"
        ok = torch.tensor([0 if (why or any(w for _, w in allh)) else 1], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        self._peer_bases = list(opened.keys())
        if int(ok.item()) == 0:
            self.peer_fallback = why or next((w for _, w in allh if w), "another rank could not map peer memory")
            self._peer_close()
            self.grad_comm = "fp32"
            return
        self._peer = g
        self._peer_ptrs = tuple(t.data_ptr() for t in bufs.values())
        plan, so = [], 0
        for _, a, b in self.buckets:
            runs = []
            for x, y in self._bucket_runs(a, b):
                x0, x1 = peer_partition(x, y, world, rank)
                if x1 > x0:
                    runs.append((x0, x1 - x0, so))
                    so += x1 - x0
            plan.append(runs)
        assert len(plan) <= 32, "more gradient buckets than flag slots"
        self._peer_plan = plan
        self.exp_avg = torch.zeros(max(so, 4), dtype=torch.float32, device=dev)
        self.exp_avg_sq = torch.zeros(max(so, 4), dtype=torch.float32, device=dev)
        import os as _os
        self._peer_ctas = int(_os.environ.get("ETP_PEER_CTAS", "64"))
        self._peer_write_reduced = 0
        dist.barrier()

    def _peer_close(self):
        for r, hb in self._peer_bases:
            try:
                _ipc_release(r, hb)
            except Exception:  # noqa: BLE001 - interpreter shutdown
                pass
        self._peer_bases = []

    def __del__(self):
        if getattr(self, "_peer_bases", None):
            self._peer_close()

    def owned_ranges(self):
        """[(a, b)] relative to the trainer's slice: what this rank reduces and updates (everything, unless peer mode)."""
        if self._peer is None:
            return [(0, self.hi - self.lo)]
        return [(x0 - self.lo, x0 - self.lo + n) for runs in self._peer_plan for x0, n, _ in runs]

    def peer_error(self):
        """0, or 1 + kind of a flag wait that gave up (synchronises the device)."""
        if self._peer is None:
            return 0
        v = i32(0)
        _L._check(_L.lib().etp_peer_error(C.byref(v)), "etp_peer_error")
        return int(v.value)

    def _join_after_update(self, main):
        """End of optimizer_step: a pipelined step() makes the compute stream wait for the navigation buckets only (the next
        step's first kernels read those weights; its panorama branch, on its own stream, waits for the rest)."""
        if self._pipelined and self._k_nav >= 0 and self._k_nav < len(self.buckets) - 1:
            main.wait_event(self._ev_nav)
            self._pending_join = True
        else:
            main.wait_stream(self.side)
            self._pending_join = False

    def _optimizer_step_peer(self):
        m, L0, g = self.m, _L.lib(), C.byref(self._peer)
        if (m._direct_grad.data_ptr(), m._flat.data_ptr(), m._flat_bf16.data_ptr()) != self._peer_ptrs[:3]:
            raise RuntimeError("the flat buffers moved after the peer group was built (rebuild the trainer)")
        main = torch.cuda.current_stream()
        side_ptr = C.c_void_p(self.side.cuda_stream)
        X, t, nb = m.config.num_x_layers, self.t, len(self.buckets)
        gsl = m._direct_grad[self.lo:self.hi]

        def finish(bi):
            # nobody may clear (or, next step, accumulate into) a gradient slice before EVERY owner has read it, nor read a
            # bucket's weights before every owner has written them: DONE of all ranks, then the slice is cleared right here
            _L._check(L0.etp_peer_wait(g, 1, bi, bi + 1, t, 30.0, side_ptr), "etp_peer_wait")
            if self._clear_after_update:
                with torch.cuda.stream(self.side):
                    gsl[self.buckets[bi][1]:self.buckets[bi][2]].zero_()

        for bi, (nm, a, b) in enumerate(self.buckets):
            if nm.startswith("x_layer_") or nm == "nav_head" or nm.startswith("pano_layer_"):
                ev = (self._pano_events[int(nm.split("_")[-1])] if nm.startswith("pano_layer_") else
                      self._events[X if nm == "nav_head" else int(nm.split("_")[-1])])
                _L._check(L0.etp_stream_wait_event(side_ptr, C.c_void_p(ev)), "etp_stream_wait_event")
            else:
                self.side.wait_stream(main)
                if self.pano_stream is not None:
                    self.side.wait_stream(self.pano_stream)
            _L._check(L0.etp_peer_signal(g, 0, bi, t, side_ptr), "etp_peer_signal")
            _L._check(L0.etp_peer_wait(g, 0, bi, bi + 1, t, 30.0, side_ptr), "etp_peer_wait")
            for x0, n, so in self._peer_plan[bi]:
                _L._check(L0.etp_peer_reduce_adamw(
                    g, x0, n, C.c_void_p(self.exp_avg.data_ptr() + 4 * so), C.c_void_p(self.exp_avg_sq.data_ptr() + 4 * so),
                    self.lr, self.betas[0], self.betas[1], self.eps, self.wd, t, self._peer_write_reduced, self._peer_ctas,
                    side_ptr), "etp_peer_reduce_adamw")
            _L._check(L0.etp_peer_signal(g, 1, bi, t, side_ptr), "etp_peer_signal")
            # the previous bucket is finished one bucket late (its owners had the time of this bucket's kernel to get done);
            # the last bucket of the navigation group and the very last one are finished at once
            if bi > 0 and bi - 1 != self._k_nav:
                finish(bi - 1)
            if bi == self._k_nav or bi == nb - 1:
                finish(bi)
            if bi == self._k_nav:
                self._ev_nav.record(self.side)
        if self._clear_after_update and m._tok_scratch is not None:
            with torch.cuda.stream(self.side):
                m._tok_scratch.zero_()
        self._join_after_update(main)
        m._bf16_fresh = True

    @staticmethod
    def _active_ranges(model, lo, hi):
        """Maximal runs [a, b) of the flat layout inside [lo, hi) whose parameters all require a gradient (the alignment
        padding between two trainable tensors is part of the run: it holds zeros and stays zero)."""
        ents = sorted((off, off + numel, model._pmap[name].requires_grad)
                      for name, (off, numel, _) in model.layout.entries.items() if lo <= off < hi)
        runs, cur = [], None
        for i, (a, b, req) in enumerate(ents):
            nxt = ents[i + 1][0] if i + 1 < len(ents) else hi
            if req:
                cur = [a, nxt] if cur is None else [cur[0], nxt]
            elif cur is not None:
                cur[1] = a
                runs.append(tuple(cur))
                cur = None
        if cur is not None:
            runs.append((cur[0], hi))
        return runs

    def join(self):
        """Make the current stream wait for everything a pipelined step() left running on the update stream (the panorama
        buckets' exchange / AdamW).  Call it before reading parameters or gradients, evaluating, or checkpointing."""
        if self.side is not None:
            torch.cuda.current_stream().wait_stream(self.side)
        self._pending_join = False

    def zero_grad(self):
        if self._pending_join:
            self.join()
        self._grads_clean = False
        self.m._direct_grad[self.lo:self.hi].zero_()
        if self.m._tok_scratch is not None:
            self.m._tok_scratch.zero_()

    def forward_backward(self, d):
        if self.pano_stream is not None and self.overlap:
            return self._forward_backward_overlapped(d)
        if self._pending_join:
            self.join()
        m = self.m
        pano, pmask = m.forward_panorama(d["rgb_fts"], d["dep_fts"], d["loc_fts"], d["nav_types"], d["view_lens"])
        # the trainer feeds the masked mean of the view embeddings back into the map as a node feature
        # (ss_trainer_ETP.py:838-839, graph_utils.py:206): here it is added to node 1 so the panorama branch trains
        w = pmask.unsqueeze(-1).float()
        avg = (pano * w).sum(1) / w.sum(1)
        img = d["gmap_img_fts"].clone()
        img[:, 1] = img[:, 1] + avg
        nav = m.forward_navigation(d["txt_embeds"], d["txt_masks"], None, d["gmap_step_ids"], img, d["gmap_pos_fts"],
                                   d["gmap_masks"], d["gmap_visited_masks"], d["gmap_pair_dists"])
        logits = nav["global_logits"]
        # caller-side loss (ss_trainer_ETP.py:890-892: CE, sum over the batch, ignore_index=-100; :1055 divides by the
        # number of actions) fused with its gradient and the greedy action: one kernel instead of torch's softmax /
        # nll / nan_to_num chain; the gradient enters autograd at the logits
        loss_sum, dlogits, self.last_action, _ = _L.step_loss(logits, d["labels"], grad_scale=1.0 / logits.shape[0])
        logits.backward(dlogits)
        return logits, loss_sum / logits.shape[0]

    def _persistent(self, name, like):
        buf = self._bufs.get(name)
        if buf is None or buf.shape != like.shape or buf.device != like.device:
            buf = torch.empty(like.shape, dtype=torch.float32, device=like.device)
            self._bufs[name] = buf
        return buf

    def _forward_backward_overlapped(self, d):
        """The same step with the panorama branch on its OWN stream.  Its 768 view rows keep ~130 SMs idle whatever the
        kernel; the only node-independent GEMMs of the navigation call are the instruction's all-layer K|V projection
        (forward) and its weight gradient (backward).  So: forward_panorama (and the masked mean into the map feature)
        runs next to the K|V projection, which leaves ``pano_sms`` SMs free (etp_nav_inputs.side_sm_reserve,
        img_ready_event); backward_panorama starts as soon as d_gmap_img_fts is final (img_grad_event) and runs next to
        the text-side weight gradient.  No autograd graph is built: the step-level C calls are issued directly, in the
        order and with the dropout seeds forward_backward() uses (same results)."""
        m = self.m
        main, S2 = torch.cuda.current_stream(), self.pano_stream
        L0, s2_ptr = _L.lib(), C.c_void_p(self.pano_stream.cuda_stream)
        m._refresh_cache()
        rgb, dep, loc = _f32c(d["rgb_fts"]), _f32c(d["dep_fts"]), _f32c(d["loc_fts"])
        nt, vl = d["nav_types"].contiguous().long(), d["view_lens"].contiguous().long()
        aux = (m._mask_u8(d["txt_masks"]), d["gmap_step_ids"].contiguous().long(), _f32c(d["gmap_pos_fts"]),
               m._mask_u8(d["gmap_masks"]), m._mask_u8(d["gmap_visited_masks"]), _f32c(d["gmap_pair_dists"]))
        txt, img_in = _txtc(d["txt_embeds"]), _f32c(d["gmap_img_fts"])
        drop_p, drop_n = m._next_dropout(), m._next_dropout()     # panorama call first, as in forward_backward()
        # ---- forward: panorama branch on S2, navigation on the compute stream
        S2.wait_stream(main)
        if self._pending_join:      # pipelined step(): the panorama weights / gradient slices are final when the update stream is
            S2.wait_stream(self.side)
            self._pending_join = False
        if self._debug_pano_start is not None:     # tests: when the panorama branch of this step was allowed to start
            self._debug_pano_start.record(S2)
        with torch.cuda.stream(S2):
            pano, pmask_u8, saved_p, _ = _pano_forward(m, rgb, dep, loc, nt, vl, 1, drop_p)
            w = pmask_u8.unsqueeze(-1).float()
            ws = w.sum(1)
            # the two tensors that cross streams live in buffers the trainer keeps (ordering by the events below and the
            # stream joins at the step boundaries): a per-step allocation would need record_stream(), whose deferred
            # reuse makes the caching allocator grow by one block per step the host runs ahead
            img = self._persistent("img", img_in)
            img.copy_(img_in)
            img[:, 1] = img[:, 1] + (pano * w).sum(1) / ws      # the very operations of forward_backward(): same bits
            _L._check(L0.etp_event_record(C.c_void_p(self._ev_img), s2_ptr), "etp_event_record")
        for t in (rgb, dep, loc, nt, vl):
            if t.data_ptr() not in self._seen_inputs:   # caller-owned inputs: tell the allocator once that S2 reads them
                t.record_stream(S2)
                self._seen_inputs.add(t.data_ptr())
        ni_extra = dict(img_ready_event=self._ev_img, side_sm_reserve=self.pano_sms)
        embeds, logits, saved_n, _ = _nav_forward(m, txt, img, aux, 1, drop_n, **ni_extra)
        loss_sum, dlogits, self.last_action, _ = _L.step_loss(logits, d["labels"], grad_scale=1.0 / logits.shape[0])
        # ---- backward: navigation on the compute stream; panorama on S2 from the moment d_gmap_img_fts is final
        _, d_img, _, _, _ = _nav_backward_raw(m, txt, img, aux, drop_n, saved_n, None, dlogits, False, True,
                                              img_grad_event=self._ev_dimg, side_sm_reserve=self.pano_sms,
                                              d_img_out=self._persistent("d_img", img))
        _L._check(L0.etp_stream_wait_event(s2_ptr, C.c_void_p(self._ev_dimg)), "etp_stream_wait_event")
        with torch.cuda.stream(S2):
            d_pano = w * (d_img[:, 1] / ws).unsqueeze(1)          # backward of the masked mean into node 1
            _pano_backward_raw(m, rgb, dep, loc, nt, vl, pmask_u8, drop_p, saved_p, d_pano, False, False)
        # the panorama gradients are part of this call's result: the compute stream joins (it has nothing else queued;
        # the bucketed update on the side stream is unaffected)
        main.wait_stream(S2)
        return logits, loss_sum / logits.shape[0]

    def _bucket_runs(self, a, b):
        """Trainable runs (absolute flat offsets) inside bucket [a, b) (offsets relative to self.lo)."""
        out = []
        for ra, rb in self.active:
            x, y = max(ra, self.lo + a), min(rb, self.lo + b)
            if x < y:
                out.append((x, y))
        return out

    def _adamw(self, a, b, scale, stream_ptr):
        m, o = self.m, a - self.lo
        _L._check(_L.lib().etp_adamw_step(
            C.c_void_p(m._flat.data_ptr() + 4 * a), C.c_void_p(m._flat_bf16.data_ptr() + 2 * a),
            C.c_void_p(m._direct_grad.data_ptr() + 4 * a), C.c_void_p(self.exp_avg.data_ptr() + 4 * o),
            C.c_void_p(self.exp_avg_sq.data_ptr() + 4 * o), b - a, self.lr, self.betas[0], self.betas[1], self.eps,
            self.wd, self.t, scale, stream_ptr), "etp_adamw_step")

    def optimizer_step(self):
        """Everything here is only ENQUEUED: the backward kernels are still running.  Per bucket, on the side stream: wait
        for the bucket's completion event, all-reduce it (SUM over ranks; DDP's 1/world is folded into AdamW's grad_scale),
        AdamW over its trainable runs.  The compute stream joins the side stream at the end."""
        m = self.m
        g = m._direct_grad[self.lo:self.hi]
        self.t += 1
        scale = 1.0 / self.world if self.world > 1 else 1.0
        if self.side is None:      # no device (host-logic tests with a stubbed library)
            if self.world > 1:
                from .dist import allreduce_buckets_
                allreduce_buckets_(g, self.buckets, self.world)
            for a, b in self.active:
                self._adamw(a, b, scale, _L.stream_ptr())
            m._bf16_fresh = True
            return
        if self._peer is not None:
            return self._optimizer_step_peer()
        L0 = _L.lib()
        main = torch.cuda.current_stream()
        side_ptr = C.c_void_p(self.side.cuda_stream)
        X = m.config.num_x_layers
        for bi, (nm, a, b) in enumerate(self.buckets):
            if nm.startswith("x_layer_") or nm == "nav_head" or nm.startswith("pano_layer_"):
                ev = (self._pano_events[int(nm.split("_")[-1])] if nm.startswith("pano_layer_") else
                      self._events[X if nm == "nav_head" else int(nm.split("_")[-1])])
                _L._check(L0.etp_stream_wait_event(side_ptr, C.c_void_p(ev)), "etp_stream_wait_event")
            else:
                self.side.wait_stream(main)       # final only when the whole backward is ...
                if self.pano_stream is not None:
                    self.side.wait_stream(self.pano_stream)   # ... including the panorama branch on its own stream
            with torch.cuda.stream(self.side):
                if self.world > 1:
                    import torch.distributed as dist
                    if self._comm_buf is not None:
                        c = self._comm_buf[a:b]
                        c.copy_(g[a:b])                                   # fp32 -> bf16 (round to nearest even)
                        dist.all_reduce(c, op=dist.ReduceOp.SUM)
                        g[a:b].copy_(c)                                   # back into the fp32 buffer AdamW reads
                    else:
                        dist.all_reduce(g[a:b], op=dist.ReduceOp.SUM)
                for x, y in self._bucket_runs(a, b):
                    self._adamw(x, y, scale, side_ptr)
                if self._clear_after_update:
                    g[a:b].zero_()
                if bi == self._k_nav:
                    self._ev_nav.record(self.side)
        if self._clear_after_update and m._tok_scratch is not None:
            with torch.cuda.stream(self.side):
                m._tok_scratch.zero_()
        self._join_after_update(main)
        m._bf16_fresh = True  # AdamW rewrote the flat parameters and their bf16 image (a high-precision image is now stale)

    def step(self, d, keep_grads=False, pipelined=False):
        """zero_grad + forward_backward + optimizer_step.  Unless ``keep_grads``, each bucket's gradient slice is cleared on
        the update stream right behind its update (under the rest of the backward), so the next step does not start with a
        300 MB memset on the compute stream: after step() the gradient buffer reads zero, as after the reference's
        ``optimizer.zero_grad()`` (ss_trainer_ETP.py:499).
        ``pipelined=True`` (training loops): the compute stream returns as soon as the NAVIGATION buckets are updated; the
        panorama buckets — last to finish in the backward, first to be needed by the next forward, but on the panorama
        branch's own stream — complete under the next step's instruction-side GEMM.  The caller's next call must be another
        step() / forward_backward() / zero_grad() (they pick the pending join up) or ``join()``."""
        if not self._grads_clean:
            self.zero_grad()
        logits, _ = self.forward_backward(d)
        self._clear_after_update = not keep_grads and self.side is not None
        self._pipelined = bool(pipelined) and self.overlap and self.pano_stream is not None
        self.optimizer_step()
        self._grads_clean, self._clear_after_update, self._pipelined = self._clear_after_update, False, False
        return logits



def get_vlnbert_models(config=None):
    """Replacement for ``vlnbert_init.get_vlnbert_models`` (vlnce_baselines/models/etp/vlnbert_init.py:13-66).

    ``config`` carries ``pretrained_path, task_type, use_depth_embedding, use_sprels, fix_lang_embedding,
    fix_pano_embedding`` like the reference's model config.  Checkpoint keys are remapped the same way:
    ``module.`` stripped (:24-25), then HF's ``bert.`` base-model prefix stripped (what
    ``from_pretrained(state_dict=...)`` does for the ``bert.``-prefixed pre-training keys)."""
    cfg = PlannerConfig.for_task(getattr(config, "task_type", "r2r"),
                                 use_depth_embedding=getattr(config, "use_depth_embedding", True),
                                 graph_sprels=getattr(config, "use_sprels", True),
                                 fix_lang_embedding=getattr(config, "fix_lang_embedding", False),
                                 fix_pano_embedding=getattr(config, "fix_pano_embedding", False))
    cfg.update_lang_bert = not cfg.fix_lang_embedding
    model = B200Planner(cfg)
    path = getattr(config, "pretrained_path", None)
    if path is not None:
        ckpt = torch.load(path, map_location="cpu")
        model.load_state_dict(remap_checkpoint_keys(ckpt, model.state_dict().keys()), strict=False)
    return model


def remap_checkpoint_keys(ckpt, own_keys):
    own = set(own_keys)
    out = {}
    for k, v in ckpt.items():
        if k.startswith("module."):
            k = k[7:]
        for pre in ("", "bert.", "net.vln_bert.", "net.module.vln_bert.", "vln_bert."):
            if pre and k.startswith(pre) and k[len(pre):] in own:
                k = k[len(pre):]
                break
        if k in own:
            out[k] = v
    return out
