"""Drop-in boundary: the ``endodav`` model class of the reference (models/endodav/endodav.py:52-160)
re-hosted on the sm_100a engine.

What stays byte-compatible with the reference (SURVEY.md section 8(b)):
  * the constructor keyword arguments and their defaults (endodav.py:53-73);
  * ``state_dict()`` keys, shapes and buffers (``pos_encoder.pe``), so checkpoints written by
    ``trainer_end_to_end_video.py:1094-1115`` load with ``load_state_dict`` / the key-filtering
    idiom of ``evaluate_depth_video.py:91-93``;
  * attributes ``.pretrained``, ``.head``, ``.head.motion_modules`` (trainer...:337-339);
  * ``forward(x[B,T,3,H,W]) -> {("disp", s): [B*T,1,h_s,w_s]}`` and
    ``infer_video_depth(frames[N,H,W,3] uint8) -> float32 [N,H,W]``.

What is different: the sub-modules are parameter containers only.  The arithmetic runs in
hand-written CUDA kernels behind the C ABI (include/endodav_b200.h); there is no PyTorch or
CPU fallback -- calling ``forward`` without the built library or without an sm_100 GPU raises.
Inference only (the reference's training loop is out of scope).
"""
import math
import os

import numpy as np
import torch
import torch.nn as nn

from . import engine as _engine
from . import pack as _pack
from . import video as _video

_MODEL_SIZES = {
    "vits": dict(dim=384, depth=12, heads=6, pos_tokens=37 * 37 + 1, taps=[2, 5, 8, 11]),
    "vitl": dict(dim=1024, depth=24, heads=16, pos_tokens=16 * 16 + 1, taps=[4, 11, 17, 23]),
    # endodac "base" (vision_transformer.py:368-382; endodac.py:176-199)
    "vitb": dict(dim=768, depth=12, heads=12, pos_tokens=37 * 37 + 1, taps=[8, 9, 10, 11]),
}


# -----------------------------------------------------------------------------------------
# parameter layout
# -----------------------------------------------------------------------------------------
def _lora_entries(prefix, n_in, n_out, lora_type, r):
    ents = [(prefix + ".weight", (n_out, n_in), "linear"), (prefix + ".bias", (n_out,), "zeros")]
    if lora_type == "ssb":
        ents += [(prefix + ".lora_A", (n_in, 1), "ones"), (prefix + ".lora_B", (n_out, 1), "ones")]
    elif lora_type in ("lora", "dvlora", "dash"):
        ents += [(prefix + ".lora_A", (r, n_in), "kaiming"), (prefix + ".lora_B", (n_out, r), "zeros")]
        if lora_type == "dvlora":
            ents += [(prefix + ".lora_U", (r, 1), "kaiming"), (prefix + ".lora_V", (n_out, 1), "kaiming")]
        if lora_type == "dash":
            ents += [(prefix + ".lora_index", (8,), "zeros"), (prefix + ".weight_u_top", (n_out, 8), "zeros"),
                     (prefix + ".weight_vt_top", (8, n_in), "zeros")]
    return ents


def parameter_layout(encoder, features, out_channels, num_frames, pe, r, lora_type, residual_block_indexes,
                     temporal_lora, disable_conv_head, motion=True, head_prefix="head.", include_cls_token=True, use_bn=False, use_clstoken=False):
    """Ordered ``[(state_dict key, shape, init kind)]`` reproducing the reference's checkpoint
    layout (SURVEY.md section 5).  ``init kind`` is only used for fresh random models.
    ``motion=False, head_prefix="depth_head."`` is the layout of the ``endodac`` image model
    (models/endodac/endodac.py:14-127,213-216): the same DPT head without temporal modules.
    ``include_cls_token`` does not change the layout: the reference keeps ``cls_token`` and the full ``pos_embed`` in the
    state_dict even when the forward ignores them (vision_transformer.py:170-176)."""
    sz = _MODEL_SIZES[encoder]
    D, F, oc = sz["dim"], features, list(out_channels)
    L = []
    p = "pretrained."
    L += [(p + "cls_token", (1, 1, D), "tiny"), (p + "pos_embed", (1, sz["pos_tokens"], D), "trunc02"),
          (p + "mask_token", (1, D), "zeros"), (p + "patch_embed.proj.weight", (D, 3, 14, 14), "kaiming"),
          (p + "patch_embed.proj.bias", (D,), "zeros")]
    for i in range(sz["depth"]):
        b = p + "blocks.%d." % i
        L += [(b + "norm1.weight", (D,), "ones"), (b + "norm1.bias", (D,), "zeros"),
              (b + "attn.qkv.weight", (3 * D, D), "trunc02"), (b + "attn.qkv.bias", (3 * D,), "zeros"),
              (b + "attn.proj.weight", (D, D), "trunc02"), (b + "attn.proj.bias", (D,), "zeros"),
              (b + "ls1.gamma", (D,), "ls"), (b + "norm2.weight", (D,), "ones"), (b + "norm2.bias", (D,), "zeros")]
        L += _lora_entries(b + "mlp.fc1", D, 4 * D, lora_type, r)
        L += _lora_entries(b + "mlp.fc2", 4 * D, D, lora_type, r)
        L += [(b + "ls2.gamma", (D,), "ls")]
        if i in residual_block_indexes:
            bc = D // 8
            rb = b + "residual_."
            L += [(rb + "conv1.weight", (bc, D, 1, 1), "kaiming"), (rb + "norm1.weight", (bc,), "ones"),
                  (rb + "norm1.bias", (bc,), "zeros"), (rb + "conv2.weight", (bc, bc, 3, 3), "kaiming"),
                  (rb + "norm2.weight", (bc,), "ones"), (rb + "norm2.bias", (bc,), "zeros"),
                  (rb + "conv3.weight", (D, bc, 1, 1), "kaiming"), (rb + "norm3.weight", (D,), "zeros"),
                  (rb + "norm3.bias", (D,), "zeros")]
    L += [(p + "norm.weight", (D,), "ones"), (p + "norm.bias", (D,), "zeros")]
    h = head_prefix
    for i in range(4):
        L += [(h + "projects.%d.weight" % i, (oc[i], D, 1, 1), "kaiming"), (h + "projects.%d.bias" % i, (oc[i],), "zeros")]
    L += [(h + "resize_layers.0.weight", (oc[0], oc[0], 4, 4), "kaiming"), (h + "resize_layers.0.bias", (oc[0],), "zeros"),
          (h + "resize_layers.1.weight", (oc[1], oc[1], 2, 2), "kaiming"), (h + "resize_layers.1.bias", (oc[1],), "zeros"),
          (h + "resize_layers.3.weight", (oc[3], oc[3], 3, 3), "kaiming"), (h + "resize_layers.3.bias", (oc[3],), "zeros")]
    if use_clstoken:   # dpt.py:92-99, registered between resize_layers and scratch
        for i in range(4):
            L += [(h + "readout_projects.%d.0.weight" % i, (D, 2 * D), "linear"), (h + "readout_projects.%d.0.bias" % i, (D,), "zeros")]
    s = h + "scratch."
    for i in range(4):
        L += [(s + "layer%d_rn.weight" % (i + 1), (F, oc[i], 3, 3), "kaiming")]
    for k in range(1, 5):
        rn = s + "refinenet%d." % k
        L += [(rn + "out_conv.weight", (F, F, 1, 1), "kaiming"), (rn + "out_conv.bias", (F,), "zeros")]
        for u in (1, 2):
            for c in (1, 2):
                L += [(rn + "resConfUnit%d.conv%d.weight" % (u, c), (F, F, 3, 3), "kaiming"),
                      (rn + "resConfUnit%d.conv%d.bias" % (u, c), (F,), "zeros")]
            if use_bn:   # registration order of ResidualConvUnit.__init__ (util/blocks.py:49-59): conv1, conv2, bn1, bn2
                for c in (1, 2):
                    b = rn + "resConfUnit%d.bn%d." % (u, c)
                    L += [(b + "weight", (F,), "ones"), (b + "bias", (F,), "zeros"), (b + "running_mean", (F,), "buffer_zeros"),
                          (b + "running_var", (F,), "buffer_ones"), (b + "num_batches_tracked", (), "buffer_count")]
    if disable_conv_head:
        L += [(s + "output_conv1.weight", (F // 2, F, 3, 3), "kaiming"), (s + "output_conv1.bias", (F // 2,), "zeros"),
              (s + "output_conv2.0.weight", (32, F // 2, 3, 3), "kaiming"), (s + "output_conv2.0.bias", (32,), "zeros"),
              (s + "output_conv2.2.weight", (1, 32, 1, 1), "kaiming"), (s + "output_conv2.2.bias", (1,), "zeros")]
    for j, C in enumerate([oc[2], oc[3], F, F] if motion else []):
        t = h + "motion_modules.%d.temporal_transformer." % j
        L += [(t + "norm.weight", (C,), "ones"), (t + "norm.bias", (C,), "zeros"),
              (t + "proj_in.weight", (C, C), "kaiming"), (t + "proj_in.bias", (C,), "zeros")]
        tb = t + "transformer_blocks.0."
        for a in range(2):
            ab = tb + "attention_blocks.%d." % a
            L += [(ab + "to_q.weight", (C, C), "kaiming"), (ab + "to_k.weight", (C, C), "kaiming"),
                  (ab + "to_v.weight", (C, C), "kaiming"), (ab + "to_out.0.weight", (C, C), "kaiming"),
                  (ab + "to_out.0.bias", (C,), "zeros")]
            if pe == "ape":
                L += [(ab + "pos_encoder.pe", (1, num_frames, C), "buffer_pe")]
        for a in range(2):
            L += [(tb + "norms.%d.weight" % a, (C,), "ones"), (tb + "norms.%d.bias" % a, (C,), "zeros")]
        L += [(tb + "ff.net.0.proj.weight", (8 * C, C), "kaiming"), (tb + "ff.net.0.proj.bias", (8 * C,), "zeros")]
        L += _lora_entries(tb + "ff.net.2", 4 * C, C, lora_type if temporal_lora else "none", r)
        L += [(tb + "ff_norm.weight", (C,), "ones"), (tb + "ff_norm.bias", (C,), "zeros"),
              (t + "proj_out.weight", (C, C), "zeros"), (t + "proj_out.bias", (C,), "zeros")]  # zero_module, motion_module.py:57-58
    if not disable_conv_head:
        for k in range(1, 5):
            c = h + "conv_depth_%d.head." % k
            L += [(c + "0.weight", (F // 2, F, 3, 3), "kaiming"), (c + "0.bias", (F // 2,), "zeros"),
                  (c + "2.weight", (32, F // 2, 3, 3), "kaiming"), (c + "2.bias", (32,), "zeros"),
                  (c + "4.weight", (1, 32, 1, 1), "kaiming"), (c + "4.bias", (1,), "zeros")]
    return L


def _init_tensor(shape, kind):
    if kind == "zeros":
        return torch.zeros(shape)
    if kind == "ones":
        return torch.ones(shape)
    if kind == "ls":
        return torch.full(shape, 1e-5)  # LayerScale init_values (vision_transformer.py:360)
    if kind == "tiny":
        return torch.randn(shape) * 1e-6
    if kind == "trunc02":
        return nn.init.trunc_normal_(torch.empty(shape), std=0.02)
    if kind in ("kaiming", "linear"):
        t = torch.empty(shape)
        if t.dim() < 2:
            return t.zero_()
        return nn.init.kaiming_uniform_(t, a=math.sqrt(5))
    raise ValueError(kind)


def _sinusoid(d_model, max_len):
    position = torch.arange(max_len).unsqueeze(1)
    div_term = torch.exp(torch.arange(0, d_model, 2) * (-math.log(10000.0) / d_model))
    pe = torch.zeros(1, max_len, d_model)
    pe[0, :, 0::2] = torch.sin(position * div_term)
    pe[0, :, 1::2] = torch.cos(position * div_term)
    return pe


class _Holder(nn.Module):
    """Parameter container mirroring one reference sub-module; holds weights, computes nothing."""

    def forward(self, *a, **k):  # pragma: no cover
        raise RuntimeError("endodav_b200 sub-modules are parameter containers; call the top-level model")


def _attach(root, key, tensor, is_buffer):
    parts = key.split(".")
    mod = root
    for i, name in enumerate(parts[:-1]):
        nxt = mod._modules.get(name)
        if nxt is None:
            nxt = _Holder()
            mod.add_module(name, nxt)
        mod = nxt
    if is_buffer:
        mod.register_buffer(parts[-1], tensor)
    else:
        mod.register_parameter(parts[-1], nn.Parameter(tensor, requires_grad=False))


def _listify(mod):
    """Containers whose children are all integer-named behave like nn.ModuleList (indexable)."""
    for name, child in list(mod._modules.items()):
        _listify(child)
        names = list(child._modules.keys())
        if names and all(n.isdigit() for n in names) and not child._parameters and not child._buffers:
            ml = nn.ModuleList()
            # keep sparse indices (resize_layers has no '2', output_conv2 no '1') addressable by key
            dense = names == [str(i) for i in range(len(names))]
            if dense:
                for n in names:
                    ml.append(child._modules[n])
                mod._modules[name] = ml


class endodav(nn.Module):
    INFER_LEN = _video.INFER_LEN
    OVERLAP = _video.OVERLAP
    KEYFRAMES = _video.KEYFRAMES
    INTERP_LEN = _video.INTERP_LEN

    def __init__(
        self,
        encoder='vitl',
        features=256,
        out_channels=[256, 512, 1024, 1024],
        use_bn=False,
        use_clstoken=False,
        num_frames=32,
        pe='ape',
        # endodav settings
        r=4,
        image_shape=(224, 280),
        lora_type="lora",
        pretrained_path=None,
        residual_block_indexes=[],
        include_cls_token=True,
        inv_sigmoid=False,
        temporal_lora=False,
        disable_conv_head=False,
        out_sigmoid=False,
        # endodav_b200 extension (keyword-only in spirit): compute dtype of the CUDA path
        dtype=None,
    ):
        super().__init__()
        if encoder not in _MODEL_SIZES:
            raise KeyError(encoder)  # the reference indexes its backbone table the same way (endodav.py:80-91)
        if lora_type not in ("none", "lora", "dvlora", "ssb", "dash"):
            raise ValueError("unknown lora_type %r" % (lora_type,))
        if pe not in ("ape", "rope"):
            raise NotImplementedError(pe)
        self.encoder = encoder
        self.image_shape = tuple(image_shape)
        self.r = r
        self.intermediate_layer_idx = {'vits': [2, 5, 8, 11], 'vitl': [4, 11, 17, 23]}
        self._cfg = dict(encoder=encoder, features=features, out_channels=list(out_channels), num_frames=num_frames,
                         pe=pe, r=r, lora_type=lora_type, residual_block_indexes=list(residual_block_indexes),
                         temporal_lora=temporal_lora, disable_conv_head=disable_conv_head,
                         include_cls_token=bool(include_cls_token), use_bn=bool(use_bn), use_clstoken=bool(use_clstoken))
        self._inv_sigmoid = bool(inv_sigmoid)
        self._out_sigmoid = bool(out_sigmoid)
        self._dtype_name = (dtype or os.environ.get("ENDODAV_DTYPE", "fp16")).lower()
        if self._dtype_name not in _engine.DTYPES:
            raise ValueError("dtype must be one of %s" % sorted(_engine.DTYPES))
        self._engine_kind = {"tc": _engine.ENGINE_TC, "simt": _engine.ENGINE_SIMT}[os.environ.get("ENDODAV_ENGINE", "tc").lower()]
        for key, shape, kind in parameter_layout(**self._cfg):
            if kind == "buffer_pe":
                _attach(self, key, _sinusoid(shape[2], shape[1]), True)
            elif kind in ("buffer_zeros", "buffer_ones", "buffer_count"):   # BatchNorm running statistics (use_bn=True)
                _attach(self, key, torch.zeros(shape) if kind == "buffer_zeros" else torch.ones(shape) if kind == "buffer_ones"
                        else torch.tensor(0, dtype=torch.long), True)
            else:
                _attach(self, key, _init_tensor(shape, kind), False)
        _listify(self)
        self._eng = None
        self._packed_versions = None
        self._pos_key = None
        if pretrained_path is not None:
            print("load pretrained weight from {}\n".format(pretrained_path))
            path = os.path.join(pretrained_path, "video_depth_anything_{}.pth".format(self.encoder))
            self.load_state_dict(torch.load(path, map_location="cpu"), strict=False)

    # -- engine plumbing --------------------------------------------------------------------
    def _edv_config(self):
        sz = _MODEL_SIZES[self.encoder]
        c = _engine.EdvConfig()
        c.dim, c.depth, c.heads = sz["dim"], sz["depth"], sz["heads"]
        for i in range(4):
            c.taps[i] = (self._cfg.get("taps") or sz["taps"])[i]
            c.out_channels[i] = self._cfg["out_channels"][i]
        c.features = self._cfg["features"]
        c.num_frames = self._cfg["num_frames"]
        c.conv_head = 0 if self._cfg["disable_conv_head"] else 1
        c.out_sigmoid = int(self._out_sigmoid)
        c.inv_sigmoid = int(self._inv_sigmoid)
        rb = 0
        for i in self._cfg["residual_block_indexes"]:
            rb |= 1 << i
        c.res_blocks = rb
        c.rope = 1 if self._cfg["pe"] == "rope" else 0
        c.dtype = _engine.DTYPES[self._dtype_name]
        c.engine = self._engine_kind
        c.no_motion = 0 if self._cfg.get("motion", True) else 1
        c.no_normalize = 0 if getattr(self, "_normalize", True) else 1
        c.no_cls = 0 if self._cfg.get("include_cls_token", True) else 1
        c.use_clstoken = 1 if self._cfg.get("use_clstoken", False) else 0
        return c

    def _pack_state_dict(self):
        """state_dict under the key names pack.py reads (the endodav layout)."""
        return self.state_dict()

    def _versions(self):
        # (storage pointer, in-place version counter) of every parameter / buffer.  The tensor list is cached: walking
        # ~300 holder modules costs more than a 224x280 forward; `_apply` (.cuda() / .to()) and load_state_dict reset it.
        ts = self.__dict__.get("_tensor_cache")
        if ts is None:
            ts = list(self.parameters()) + list(self.buffers())
            self.__dict__["_tensor_cache"] = ts
        return tuple((p.data_ptr(), p._version) for p in ts)

    def invalidate_weights(self):
        """Force a re-pack of the weights on the next forward.

        Re-packing is triggered automatically by ``load_state_dict``, by ``.to()`` / ``.cuda()`` and by in-place
        parameter updates that bump the autograd version counter (``p.add_(...)``, ``p.copy_(...)``, optimiser steps).
        Writes through ``p.data`` (``p.data.copy_(w)``, ``p.data += ...`` -- the idiom of the reference's LoRA merge code)
        bump neither the counter nor the pointer: call this method after them."""
        self._packed_versions = None
        self.__dict__["_tensor_cache"] = None
        return self

    def _apply(self, fn, *a, **k):
        out = super()._apply(fn, *a, **k)
        self.invalidate_weights()
        return out

    def load_state_dict(self, *a, **k):
        out = super().load_state_dict(*a, **k)
        self.invalidate_weights()
        return out

    def _device(self):
        return next(self.parameters()).device

    def _ensure_engine(self, ph, pw):
        dev = self._device()
        if dev.type != "cuda":
            raise _engine.EndoDAVError(
                "endodav_b200 has no CPU path: move the model to a CUDA device first (model.cuda()); got %s" % dev)
        if self._eng is None or self._eng.device != dev:
            self._eng = _engine.Engine(self._edv_config(), dev)
            self._packed_versions = None
            self._pos_key = None
        ver = self._versions()
        if ver != self._packed_versions:
            sd = self._pack_state_dict()
            tdt = _engine.TORCH_DTYPE[_engine.DTYPES[self._dtype_name]]
            self._eng.set_weights(_pack.pack_state_dict(sd, self._cfg, tdt))
            self._packed_versions = ver
            self._pos_key = None
        if self._pos_key != (ph, pw):
            self._eng.set_weights(_pack.pos_tables(self._pack_state_dict(), self._cfg, ph, pw))
            self._pos_key = (ph, pw)
        return self._eng

    def set_compute_dtype(self, dtype):
        """'fp16' (default), 'bf16' or 'fp32' -- see DESIGN.md for the accuracy of each."""
        dtype = dtype.lower()
        if dtype not in _engine.DTYPES:
            raise ValueError(dtype)
        if _engine.DTYPES[dtype] != _engine.DTYPES[self._dtype_name]:
            self._dtype_name = dtype
            self._eng = None
        return self

    # -- reference API ------------------------------------------------------------------------
    @torch.no_grad()
    def forward(self, x):
        """endodav.forward (endodav.py:150-160): x [B,T,3,H,W] float in [0,1] ->
        {("disp", s): [B*T,1,h_s,w_s]}, s = 0..3."""
        if x.dim() != 5 or x.shape[2] != 3:
            raise ValueError("expected [B,T,3,H,W], got %s" % (tuple(x.shape),))
        B, T, _, H, W = x.shape
        h, w = self.image_shape
        assert h % 14 == 0, f"Input image height {h} is not a multiple of patch height 14"   # patch_embed.py:72
        assert w % 14 == 0, f"Input image width {w} is not a multiple of patch width: 14"    # patch_embed.py:73
        eng = self._ensure_engine(h // 14, w // 14)
        x = x.to(device=eng.device, dtype=torch.float32).contiguous()
        with torch.cuda.device(eng.device):
            eng.plan(B, T, H, W, h, w)
            disp, _ = eng.forward(x)
        return {("disp", s): disp[s] for s in range(4)}

    @torch.no_grad()
    def infer_video_depth(self, frames, input_size=518, device='cuda'):
        """endodav.infer_video_depth (endodav.py:162-254).  ``input_size`` is ignored exactly as in
        the reference (:164-174).  Uses every visible rank when torch.distributed is initialised."""
        return _video.infer_video_depth(self, frames, device=device)


class endodac(endodav):
    """Drop-in for the reference's image model ``endodac`` (models/endodac/endodac.py:144-272):
    the same DINOv2 encoder (+ LoRA / DV-LoRA MLP adapters) and DPT head as ``endodav`` without the
    temporal modules, checkpoint keys under ``pretrained.*`` / ``depth_head.*``.  It runs on the
    same sm_100a engine (``edv_config.no_motion``); SURVEY.md section 8(f) row 2.

    Kept from the reference: constructor keywords and defaults (:153-165), the size tables
    (:171-199), ``forward(pixel_values[B,3,H,W] or [B,T,3,H,W]) -> {("disp", s)}`` (:246-259) and
    ``infer_video_depth(frames, batch_size=8)`` (:261-272)."""

    _SIZES = {  # endodac.py:171-199
        "small": dict(encoder="vits", features=64, out_channels=[48, 96, 192, 384]),
        "base": dict(encoder="vitb", features=128, out_channels=[96, 192, 384, 768]),
    }

    def __init__(
        self,
        backbone_size="base",
        r=4,
        image_shape=(224, 280),
        lora_type="lora",
        pretrained_path=None,
        residual_block_indexes=[],
        include_cls_token=True,
        use_cls_token=False,
        use_bn=False,
        pre_norm=False,
        inv_sigmoid=False,
        disable_conv_head=False,
        dtype=None,
    ):
        nn.Module.__init__(self)
        assert r > 0                                       # endodac.py:168
        if backbone_size not in self._SIZES:
            raise KeyError(backbone_size)                  # the reference indexes its tables the same way (:200-204)
        if lora_type not in ("none", "lora", "dvlora"):
            # endodac.py:213-224 installs adapters only for these; any other string leaves plain linears
            lora_type = "none"
        sz = self._SIZES[backbone_size]
        self.backbone_size = backbone_size
        self.encoder = sz["encoder"]
        self.embedding_dim = _MODEL_SIZES[self.encoder]["dim"]
        self.image_shape = tuple(image_shape)
        self.r = r
        self._cfg = dict(encoder=self.encoder, features=sz["features"], out_channels=list(sz["out_channels"]),
                         num_frames=32, pe="ape", r=r, lora_type=lora_type,
                         residual_block_indexes=list(residual_block_indexes), temporal_lora=False,
                         disable_conv_head=disable_conv_head, motion=False, include_cls_token=bool(include_cls_token),
                         use_clstoken=bool(use_cls_token), use_bn=bool(use_bn))   # endodac.py:161-163 (its keyword is use_cls_token)
        # forward taps get_intermediate_layers(x, 4): the LAST four blocks (endodac.py:254;
        # vision_transformer.py:292-293), not the [2,5,8,11] table at endodac.py:183-186
        depth = _MODEL_SIZES[self.encoder]["depth"]
        self._cfg["taps"] = list(range(depth - 4, depth))
        # LoraLinear(..., r=r) keeps lora_alpha=1 here: scaling 1/r, not endodav's 2 (endodac.py:222-223)
        self._cfg["lora_scale"] = 1.0 / r
        self._normalize = bool(pre_norm)                   # endodac.py:208-211: identity unless pre_norm
        self._inv_sigmoid = bool(inv_sigmoid)
        self._out_sigmoid = False
        self._dtype_name = (dtype or os.environ.get("ENDODAV_DTYPE", "fp16")).lower()
        if self._dtype_name not in _engine.DTYPES:
            raise ValueError("dtype must be one of %s" % sorted(_engine.DTYPES))
        self._engine_kind = {"tc": _engine.ENGINE_TC, "simt": _engine.ENGINE_SIMT}[os.environ.get("ENDODAV_ENGINE", "tc").lower()]
        for key, shape, kind in parameter_layout(head_prefix="depth_head.", **{k: v for k, v in self._cfg.items() if k not in ("taps", "lora_scale")}):
            if kind in ("buffer_zeros", "buffer_ones", "buffer_count"):   # BatchNorm running statistics (use_bn=True)
                _attach(self, key, torch.zeros(shape) if kind == "buffer_zeros" else torch.ones(shape) if kind == "buffer_ones"
                        else torch.tensor(0, dtype=torch.long), True)
            else:
                _attach(self, key, _init_tensor(shape, kind), False)
        _listify(self)
        self._eng = None
        self._packed_versions = None
        self._pos_key = None
        if pretrained_path is not None:
            arch = {"small": "v2_vits", "base": "v2_vitb"}[backbone_size]   # endodac.py:177-182
            path = os.path.join(pretrained_path, "depth_anything_{}.pth".format(arch))
            self.load_state_dict(torch.load(path, map_location="cpu"), strict=False)
            print("load pretrained weight from {}\n".format(path))

    def _pack_state_dict(self):
        return {("head." + k[len("depth_head."):] if k.startswith("depth_head.") else k): v
                for k, v in self.state_dict().items()}

    @torch.no_grad()
    def forward(self, pixel_values):
        """endodac.forward (endodac.py:246-259): [B,3,H,W] (or [B,T,3,H,W], flattened) in [0,1] ->
        {("disp", s): [B,1,h_s,w_s]}."""
        if pixel_values.dim() == 5:
            pixel_values = pixel_values.flatten(0, 1)
        if pixel_values.dim() != 4 or pixel_values.shape[1] != 3:
            raise ValueError("expected [B,3,H,W], got %s" % (tuple(pixel_values.shape),))
        Bn, _, H, W = pixel_values.shape
        h, w = self.image_shape
        assert h % 14 == 0, f"Input image height {h} is not a multiple of patch height 14"
        assert w % 14 == 0, f"Input image width {w} is not a multiple of patch width: 14"
        eng = self._ensure_engine(h // 14, w // 14)
        x = pixel_values.to(device=eng.device, dtype=torch.float32).contiguous()
        with torch.cuda.device(eng.device):
            eng.plan(Bn, 1, H, W, h, w)
            disp, _ = eng.forward(x)
        return {("disp", s): disp[s] for s in range(4)}

    @torch.no_grad()
    def infer_video_depth(self, frames, batch_size=8, device='cuda'):
        """endodac.infer_video_depth (endodac.py:261-272): independent chunks of ``batch_size`` frames,
        each resized back to the frame size (bilinear, align_corners=True).  The uint8 -> float32/255
        CHW conversion and the final resize run in the library's kernels.  A CUDA uint8 tensor of any positive strides is
        read in place and gives a float32 tensor on its device (the contract of ``endodav.infer_video_depth``)."""
        frames_dev = _video.frames_device(frames, device)
        if frames_dev is None:
            frames = np.ascontiguousarray(frames)
            if frames.ndim != 4 or frames.shape[-1] != 3 or frames.dtype != np.uint8:
                raise ValueError("frames must be uint8 [N,H,W,3]")
        elif self._device() != frames_dev:
            self.to(frames_dev)
        N, H, W, _ = frames.shape
        h, w = self.image_shape
        eng = self._ensure_engine(h // 14, w // 14)
        if frames_dev is not None:
            # one input and one resized buffer for every chunk: the forward's captured CUDA graph, keyed by their
            # pointers, is replayed
            out = torch.empty(N, H, W, dtype=torch.float32, device=frames_dev)
            B = min(batch_size, N)
            x_buf = torch.empty(B, 3, H, W, dtype=torch.float32, device=frames_dev)
            r_buf = torch.empty(B, H, W, dtype=torch.float32, device=frames_dev)
            with torch.cuda.device(frames_dev):
                for c0 in range(0, N, batch_size):
                    n = min(batch_size, N - c0)
                    x = _engine.op_cubic_resize_u8(frames, H, W, out=x_buf[:n], index=np.arange(c0, c0 + n))
                    eng.plan(n, 1, H, W, h, w)
                    eng.forward(x, resize_to=(H, W), want_pyramid=False, resized_out=r_buf[:n])
                    out[c0:c0 + n].copy_(r_buf[:n])
            return out
        out = np.empty((N, H, W), dtype=np.float32)
        with torch.cuda.device(eng.device):
            for c0 in range(0, N, batch_size):
                chunk = torch.from_numpy(frames[c0:c0 + batch_size]).to(eng.device)
                n = chunk.shape[0]
                # identity-size bicubic is exact (taps 0,1,0,0): this is frame.astype(float32)/255 in CHW
                x = _engine.op_cubic_resize_u8(chunk, H, W)
                eng.plan(n, 1, H, W, h, w)
                _, resized = eng.forward(x, resize_to=(H, W), want_pyramid=False)
                out[c0:c0 + n] = resized.cpu().numpy()
        return out
