"""TEST INFRASTRUCTURE ONLY -- generate tests/golden/*.npz from the UNMODIFIED reference.

Run in the build container (needs /root/reference):

    python -m oracle.make_golden

Every fixture stores the constructor config, the weight seed, the input seed/shape and
the reference outputs; weights and inputs are regenerated from the seeds by
``oracle/weights.py`` (reference-free), so the fixtures stay small.  The reference has no
golden vectors of its own (SURVEY.md section 4, 8(c)); these files are what pins
``oracle/endodav_oracle.py`` and ``oracle/video_oracle.py``.
"""
import hashlib
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import ref_import, weights  # noqa: E402

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")

SIZES = {
    "vits": dict(features=64, out_channels=[48, 96, 192, 384]),
    "vitl": dict(features=256, out_channels=[256, 512, 1024, 1024]),
}

# name -> (ctor overrides, image_shape, input [B,T,H,W], weight seed, frame seed)
FORWARD_CASES = {
    "fwd_vits_dvlora": (dict(encoder="vits", lora_type="dvlora"), (70, 98), (1, 4, 80, 112), 1234, 4321),
    "fwd_vits_b2": (dict(encoder="vits", lora_type="dvlora"), (56, 56), (2, 3, 56, 56), 11, 12),
    "fwd_vits_lora_res_convhead": (
        dict(encoder="vits", lora_type="lora", residual_block_indexes=[2, 5, 8, 11], disable_conv_head=False),
        (224, 280), (1, 2, 224, 280), 21, 22),
    "fwd_vits_ssb_tlora": (dict(encoder="vits", lora_type="ssb", temporal_lora=True), (42, 56), (1, 3, 48, 64), 31, 32),
    "fwd_vits_dash_tlora": (dict(encoder="vits", lora_type="dash", temporal_lora=True), (42, 56), (1, 3, 48, 64), 41, 42),
    "fwd_vits_rope": (dict(encoder="vits", lora_type="dvlora", pe="rope"), (42, 56), (1, 5, 42, 56), 51, 52),
    "fwd_vitl": (dict(encoder="vitl", lora_type="dvlora"), (70, 84), (1, 2, 70, 84), 61, 62),
    # include_cls_token=False: the ViT runs on the patch tokens only (every reference script plumbs opt.include_cls_token)
    # use_bn=True: BatchNorm2d (eval mode) after both convs of every ResidualConvUnit
    "fwd_vits_bn": (dict(encoder="vits", lora_type="dvlora", use_bn=True), (42, 56), (1, 3, 48, 64), 85, 86),
    # use_clstoken=True: readout projects on [patch token | class token]; the second case takes the "class token" of a ViT
    # without one (its first patch token)
    "fwd_vits_clstoken": (dict(encoder="vits", lora_type="dvlora", use_clstoken=True), (42, 56), (1, 3, 48, 64), 87, 88),
    "fwd_vits_clstoken_nocls": (dict(encoder="vits", lora_type="lora", use_clstoken=True, include_cls_token=False), (42, 56),
                                (2, 2, 42, 56), 89, 90),
    "fwd_vits_nocls": (dict(encoder="vits", lora_type="dvlora", include_cls_token=False), (42, 56), (1, 3, 48, 64), 81, 82),
    "fwd_vits_nocls_res": (dict(encoder="vits", lora_type="lora", residual_block_indexes=[2, 5, 8, 11], include_cls_token=False),
                           (224, 280), (1, 2, 224, 280), 83, 84),
}

# Full-size BASELINE configurations (2: ViT-S 32 x 518 x 518; 4: ViT-L at 518 x 518, two frames): the reference output
# is stored as a strided sample (frames FULL_FRAMES, every FULL_STRIDE-th pixel) so the fixture stays small; it pins the
# oracle at S = 1370 tokens / T = 32 / 37x37 -> 19x19 maps, and the GPU tests compare the CUDA path with the oracle on
# the full maps.  name -> (ctor overrides, image_shape, input, weight seed, frame seed, frames kept)
FULL_CASES = {
    "full_vits_518_t32": (dict(encoder="vits", lora_type="dvlora"), (518, 518), (1, 32, 518, 518), 1234, 4321, [0, 15, 31]),
    "full_vitl_518_t2": (dict(encoder="vitl", lora_type="dvlora"), (518, 518), (1, 2, 518, 518), 61, 62, [0, 1]),
}
FULL_STRIDE = 7

VIDEO_CASES = {
    # name -> (N, H, W, image_shape, weight seed, frame seed)
    "video_n45": (45, 48, 64, (28, 42), 1234, 7),
    "video_n5": (5, 40, 56, (28, 42), 1234, 8),
}

STUB_VIDEO_N = [1, 5, 21, 22, 23, 32, 44, 45, 100]

# endodac image model (SURVEY.md 8(f)-2): name -> (reference ctor kwargs, input shape, weight seed, frame seed)
ENDODAC_CASES = {
    "dac_small_dvlora": (dict(backbone_size="small", lora_type="dvlora", image_shape=(42, 56), disable_conv_head=True),
                         (3, 3, 48, 64), 71, 72),
    "dac_small_prenorm_5d": (dict(backbone_size="small", lora_type="lora", image_shape=(56, 56), disable_conv_head=True,
                                  pre_norm=True), (2, 2, 3, 56, 56), 73, 74),
    "dac_base_lora_convhead": (dict(backbone_size="base", lora_type="lora", image_shape=(56, 70), disable_conv_head=False,
                                    inv_sigmoid=True), (2, 3, 56, 70), 75, 76),
    # the three constructor modes endodac shares with endodav: no cls token, readout projects, BatchNorm in the fusion blocks
    "dac_small_nocls_clstoken_bn": (dict(backbone_size="small", lora_type="dvlora", image_shape=(42, 56), disable_conv_head=True,
                                         include_cls_token=False, use_cls_token=True, use_bn=True), (3, 3, 42, 56), 91, 92),
    "dac_base_dvlora": (dict(backbone_size="base", lora_type="dvlora", image_shape=(70, 56), disable_conv_head=True),
                        (2, 3, 70, 56), 77, 78),
}
ENDODAC_VIDEO = {
    # name -> (ctor kwargs, N, H, W, batch_size, weight seed, frame seed)
    "dac_video_n11": (dict(backbone_size="small", lora_type="dvlora", image_shape=(28, 42), disable_conv_head=True),
                      11, 40, 56, 4, 79, 80),
}


def endodac_oracle_cfg(kw):
    return weights.endodac_cfg(kw["backbone_size"], kw.get("lora_type", "lora"), kw.get("r", 4),
                               kw.get("residual_block_indexes", []), kw.get("disable_conv_head", False),
                               kw.get("include_cls_token", True), kw.get("use_cls_token", False), kw.get("use_bn", False))


def make_endodac(manifest):
    only = [a.split("=", 1)[1] for a in sys.argv if a.startswith("--only=")]
    for name, (kw, shape, wseed, fseed) in ENDODAC_CASES.items():
        if only and name not in only:
            continue
        cfg = endodac_oracle_cfg(kw)
        sd = weights.to_endodac_keys(weights.make_state_dict(cfg, wseed))
        model = ref_import.build_reference_endodac(dict(kw, r=4))
        missing = model.load_state_dict(sd, strict=True)
        n = 1
        for d in shape[:-3]:
            n *= d
        x = weights.make_frames(1, n, shape[-2], shape[-1], fseed)[0].reshape(shape)
        with torch.no_grad():
            out = model(x)
        arrays = {"disp%d" % s: out[("disp", s)].numpy().astype(np.float32) for s in range(4)}
        np.savez_compressed(os.path.join(GOLDEN_DIR, name + ".npz"), **arrays)
        manifest[name] = dict(kind="endodac_forward", ctor={k: (list(v) if isinstance(v, tuple) else v) for k, v in kw.items()},
                              input=list(shape), weight_seed=wseed, frame_seed=fseed, keys=len(sd))
        print(name, {k: v.shape for k, v in arrays.items()}, float(arrays["disp0"].mean()), str(missing))
        if name in ("dac_small_dvlora", "dac_base_lora_convhead"):
            with open(os.path.join(GOLDEN_DIR, "state_dict_keys_%s.json" % name), "w") as f:
                json.dump([[k, list(v.shape)] for k, v in model.state_dict().items()], f)
    for name, (kw, N, H, W, bs, wseed, fseed) in ENDODAC_VIDEO.items():
        if only and name not in only:
            continue
        cfg = endodac_oracle_cfg(kw)
        sd = weights.to_endodac_keys(weights.make_state_dict(cfg, wseed))
        model = ref_import.build_reference_endodac(dict(kw, r=4))
        model.load_state_dict(sd, strict=True)
        v = weights.make_video_u8(N, H, W, fseed)
        with torch.no_grad():
            out = model.infer_video_depth(v, batch_size=bs, device="cpu")
        np.savez_compressed(os.path.join(GOLDEN_DIR, name + ".npz"), depth=out.astype(np.float32))
        manifest[name] = dict(kind="endodac_video", ctor={k: (list(v_) if isinstance(v_, tuple) else v_) for k, v_ in kw.items()},
                              input=[N, H, W], batch_size=bs, weight_seed=wseed, frame_seed=fseed)
        print(name, out.shape, float(out.mean()))


def ctor_kwargs(over, image_shape):
    enc = over.get("encoder", "vits")
    kw = dict(encoder=enc, r=4, image_shape=tuple(image_shape), disable_conv_head=True, residual_block_indexes=[])
    kw.update(SIZES[enc])
    kw.update(over)
    return kw


def oracle_cfg(kw):
    keys = ("encoder", "features", "out_channels", "num_frames", "pe", "r", "lora_type",
            "residual_block_indexes", "temporal_lora", "disable_conv_head", "include_cls_token", "use_bn", "use_clstoken")
    return weights.full_cfg({k: kw[k] for k in keys if k in kw})


def _dash_past_warmup(model):
    # DashLinear adds its SVD term only once its Python-side call counter has passed
    # warm-up (mylora/layers.py:560-582); the counter is not in the state_dict.  The
    # inference form we parity-check is the post-warm-up one, so advance the counter.
    for m in model.modules():
        if hasattr(m, "FLAG") and hasattr(m, "warmup"):
            m.FLAG = m.warmup + 1


def make_fullsize(manifest):
    import time
    for name, (over, ishape, (B, T, H, W), wseed, fseed, keep) in FULL_CASES.items():
        kw = ctor_kwargs(over, ishape)
        sd = weights.make_state_dict(oracle_cfg(kw), wseed)
        model = ref_import.build_reference_model(kw)
        model.load_state_dict(sd, strict=True)
        x = weights.make_frames(B, T, H, W, fseed)
        t0 = time.time()
        with torch.no_grad():
            out = model(x)
        d0 = out[("disp", 0)].numpy().astype(np.float32)
        arrays = {"disp0": d0[keep][:, :, ::FULL_STRIDE, ::FULL_STRIDE].copy(),
                  "disp3": out[("disp", 3)].numpy().astype(np.float32)[keep].copy(),
                  "stats": np.array([d0.mean(), d0.std(), d0.min(), d0.max()], dtype=np.float64)}
        np.savez_compressed(os.path.join(GOLDEN_DIR, name + ".npz"), **arrays)
        manifest[name] = dict(kind="forward_full", ctor={k: (list(v) if isinstance(v, tuple) else v) for k, v in kw.items()},
                              input=[B, T, H, W], weight_seed=wseed, frame_seed=fseed, frames=keep, stride=FULL_STRIDE)
        print(name, {k: v.shape for k, v in arrays.items()}, arrays["stats"], "%.1f s" % (time.time() - t0))
        del model, out


def make_metrics():
    """disp_to_depth / compute_errors of the UNMODIFIED reference on the seeded case of oracle/metrics_oracle.py."""
    import importlib.util
    import warnings

    from oracle import metrics_oracle as mo

    def load(path, name):
        spec = importlib.util.spec_from_file_location(name, os.path.join(ref_import.REFERENCE_ROOT, path))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        return mod

    layers = load("utils/layers.py", "ref_utils_layers")
    utils = load("utils/utils.py", "ref_utils_utils")
    disp, gt = mo.make_case()
    scaled, depth = layers.disp_to_depth(disp, 0.1, 150.0)
    errs = []
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for g, p in zip(gt, depth):
            p = p.copy()
            valid = np.logical_and(g > 1e-3, g < 150)
            p *= 1.0
            p[p < 1e-3] = 1e-3
            p[p > 150] = 150
            errs.append(utils.compute_errors(g, p, valid))
    np.savez_compressed(os.path.join(GOLDEN_DIR, "metrics.npz"), scaled=scaled.astype(np.float32), depth=depth.astype(np.float32),
                        errors=np.array(errs, dtype=np.float64))
    print("metrics", scaled.dtype, depth.dtype, np.array(errs)[:2])


def stub_forward(x):
    """Deterministic stand-in network used for the bit-exact index/stitch fixtures: per-frame
    disparity = channel mean + 0.1*frame-mean, so every slot's source frame is identifiable."""
    B, T, C, H, W = x.shape
    f = x.flatten(0, 1)
    d = f.mean(1, keepdim=True) + 0.1 * f.mean(dim=(1, 2, 3), keepdim=True)
    return {("disp", 0): d}


def main():
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    ref_mod = ref_import.import_reference()
    manifest = {}
    if "--metrics-only" in sys.argv:   # evaluation helpers (utils/layers.py, utils/utils.py) -> tests/golden/metrics.npz
        make_metrics()
        return
    if "--fullsize-only" in sys.argv:  # add the full-size fixtures without regenerating the others
        with open(os.path.join(GOLDEN_DIR, "manifest.json")) as f:
            manifest = json.load(f)
        make_fullsize(manifest)
        with open(os.path.join(GOLDEN_DIR, "manifest.json"), "w") as f:
            json.dump(manifest, f, indent=1)
        return
    if "--endodac-only" in sys.argv:   # add the endodac fixtures without regenerating the others
        with open(os.path.join(GOLDEN_DIR, "manifest.json")) as f:
            manifest = json.load(f)
        make_endodac(manifest)
        with open(os.path.join(GOLDEN_DIR, "manifest.json"), "w") as f:
            json.dump(manifest, f, indent=1)
        return
    only = [a.split("=", 1)[1] for a in sys.argv if a.startswith("--only=")]   # add cases without regenerating the others
    if only:
        with open(os.path.join(GOLDEN_DIR, "manifest.json")) as f:
            manifest = json.load(f)
    for name, (over, ishape, (B, T, H, W), wseed, fseed) in FORWARD_CASES.items():
        if only and name not in only:
            continue
        kw = ctor_kwargs(over, ishape)
        cfg = oracle_cfg(kw)
        sd = weights.make_state_dict(cfg, wseed)
        model = ref_import.build_reference_model(kw)
        missing = model.load_state_dict(sd, strict=True)
        _dash_past_warmup(model)
        x = weights.make_frames(B, T, H, W, fseed)
        with torch.no_grad():
            out = model(x)
        arrays = {"disp%d" % s: out[("disp", s)].numpy().astype(np.float32) for s in range(4)}
        if name in ("fwd_vits_lora_res_convhead", "fwd_vits_nocls_res"):  # keep the fixture small
            arrays["disp0"] = arrays["disp0"][:, :, ::4, ::4].copy()
            arrays["disp1"] = arrays["disp1"][:, :, ::2, ::2].copy()
        np.savez_compressed(os.path.join(GOLDEN_DIR, name + ".npz"), **arrays)
        manifest[name] = dict(kind="forward", ctor={k: (list(v) if isinstance(v, tuple) else v) for k, v in kw.items()},
                              input=[B, T, H, W], weight_seed=wseed, frame_seed=fseed,
                              keys=len(sd), params=int(sum(v.numel() for v in sd.values())))
        print(name, {k: v.shape for k, v in arrays.items()}, float(arrays["disp0"].mean()), str(missing))
        if name == "fwd_vits_dvlora":
            with open(os.path.join(GOLDEN_DIR, "state_dict_keys_vits.json"), "w") as f:
                json.dump([[k, list(v.shape)] for k, v in model.state_dict().items()], f)
        if name == "fwd_vitl":
            with open(os.path.join(GOLDEN_DIR, "state_dict_keys_vitl.json"), "w") as f:
                json.dump([[k, list(v.shape)] for k, v in model.state_dict().items()], f)
        if name == "fwd_vits_lora_res_convhead":
            with open(os.path.join(GOLDEN_DIR, "state_dict_keys_vits_lora_res_convhead.json"), "w") as f:
                json.dump([[k, list(v.shape)] for k, v in model.state_dict().items()], f)
        del model
    if only:
        with open(os.path.join(GOLDEN_DIR, "manifest.json"), "w") as f:
            json.dump(manifest, f, indent=1)
        return

    for name, (N, H, W, ishape, wseed, fseed) in VIDEO_CASES.items():
        kw = ctor_kwargs(dict(encoder="vits", lora_type="dvlora"), ishape)
        cfg = oracle_cfg(kw)
        sd = weights.make_state_dict(cfg, wseed)
        model = ref_import.build_reference_model(kw)
        model.load_state_dict(sd, strict=True)
        v = weights.make_video_u8(N, H, W, fseed)
        with torch.no_grad():
            out = model.infer_video_depth(v, device="cpu")
        np.savez_compressed(os.path.join(GOLDEN_DIR, name + ".npz"), depth=out.astype(np.float32))
        manifest[name] = dict(kind="video", ctor={k: (list(v_) if isinstance(v_, tuple) else v_) for k, v_ in kw.items()},
                              input=[N, H, W], weight_seed=wseed, frame_seed=fseed)
        print(name, out.shape, float(out.mean()))

    # bit-exact window/keyframe/stitch fixtures with a stub network
    kw = ctor_kwargs(dict(encoder="vits", lora_type="none"), (28, 42))
    model = ref_import.build_reference_model(kw)
    model.forward = stub_forward
    stub, sha = {}, {}
    for N in STUB_VIDEO_N:
        v = weights.make_video_u8(N, 30, 44, 100 + N)
        with torch.no_grad():
            d = np.ascontiguousarray(model.infer_video_depth(v, device="cpu"), dtype=np.float32)
        stub["n%d" % N] = d[:, ::2, ::2].copy()    # a strided sample keeps the file small; the digest covers every bit
        sha["n%d" % N] = hashlib.sha256(d.tobytes()).hexdigest()
    np.savez_compressed(os.path.join(GOLDEN_DIR, "video_stub.npz"), **stub)
    manifest["video_stub"] = dict(kind="video_stub", n=STUB_VIDEO_N, input=[30, 44], image_shape=[28, 42], stride=2, sha256=sha)

    make_endodac(manifest)
    make_fullsize(manifest)
    make_metrics()

    with open(os.path.join(GOLDEN_DIR, "manifest.json"), "w") as f:
        json.dump(manifest, f, indent=1)
    total = sum(os.path.getsize(os.path.join(GOLDEN_DIR, f)) for f in os.listdir(GOLDEN_DIR))
    print("golden dir bytes", total)


if __name__ == "__main__":
    main()
