"""Helpers shared by the golden-fixture tests (CPU and GPU)."""
import hashlib
import json
import os

import numpy as np

from oracle import weights

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ORACLE_KEYS = ("encoder", "features", "out_channels", "num_frames", "pe", "r", "lora_type",
               "residual_block_indexes", "temporal_lora", "disable_conv_head", "include_cls_token", "use_bn", "use_clstoken")


def manifest():
    with open(os.path.join(GOLDEN_DIR, "manifest.json")) as f:
        return json.load(f)


def load_case(name):
    m = manifest()[name]
    arrays = dict(np.load(os.path.join(GOLDEN_DIR, name + ".npz")))
    return m, arrays


def oracle_cfg(ctor):
    return weights.full_cfg({k: ctor[k] for k in ORACLE_KEYS if k in ctor})


def assert_video_stub_matches(n, got):
    """video_stub keeps, per video length n, a strided sample of the reference driver's depth and the SHA-256 of
    its full float32 bytes: the sample localises a mismatch, the digest makes the comparison bit-exact."""
    m, arrays = load_case("video_stub")
    ref = arrays["n%d" % n]
    st = m["stride"]
    assert got.dtype == np.float32 and got.shape[1:] == tuple(m["input"]), (n, got.dtype, got.shape)
    sample = got[:, ::st, ::st]
    assert sample.shape == ref.shape, (n, sample.shape, ref.shape)
    assert np.array_equal(sample, ref), (n, float(np.abs(sample - ref).max()))
    assert hashlib.sha256(np.ascontiguousarray(got).tobytes()).hexdigest() == m["sha256"]["n%d" % n], n


def subsample_like_golden(name, s, arr):
    """make_golden.py stores a strided view of the two largest maps of one case."""
    if name in ("fwd_vits_lora_res_convhead", "fwd_vits_nocls_res"):
        if s == 0:
            return arr[:, :, ::4, ::4]
        if s == 1:
            return arr[:, :, ::2, ::2]
    return arr
