"""ctypes binding of the C-ABI library (include/endodav_b200.h).

There is deliberately no fallback: if ``libendodav_b200.so`` is missing or no sm_100 GPU is
present, every entry point raises.  torch is used only for device memory and streams."""
import ctypes
import os

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "csrc", "libendodav_b200.so")

EDV_F32, EDV_BF16, EDV_F16 = 0, 1, 2
ENGINE_TC, ENGINE_SIMT = 0, 1
DTYPES = {"fp32": EDV_F32, "f32": EDV_F32, "float32": EDV_F32, "bf16": EDV_BF16, "bfloat16": EDV_BF16,
          "fp16": EDV_F16, "f16": EDV_F16, "float16": EDV_F16}
TORCH_DTYPE = {EDV_F32: torch.float32, EDV_BF16: torch.bfloat16, EDV_F16: torch.float16}

ABI_VERSION = 18  # must equal EDV_ABI_VERSION of include/endodav_b200.h (argtypes below are mirrored by hand)

EXPORTS = [
    "edv_abi_version", "edv_create", "edv_destroy", "edv_last_error", "edv_set_weight", "edv_plan", "edv_forward", "edv_forward_u8",
    "edv_output_shape", "edv_launch_count", "edv_set_debug", "edv_debug_tap", "edv_plan_buffer", "edv_set_graph_mode", "edv_graph_count", "edv_graph_status", "edv_op_gemm",
    "edv_op_attention", "edv_op_temporal_attention", "edv_op_layernorm", "edv_op_groupnorm", "edv_op_upsample",
    "edv_op_resize_f32", "edv_profile", "edv_profile_reset", "edv_profile_collect", "edv_profile_get",
    "edv_op_disp_head", "edv_op_cubic_resize_u8", "edv_op_cubic_resize_u8_gather", "edv_op_stitch_window", "edv_op_stitch_plan",
    "edv_op_disp_to_depth", "edv_op_compute_errors", "edv_op_attention_timeline", "edv_op_linear_timeline", "edv_op_linear_residual_ln",
    "edv_op_preprocess_patches", "edv_op_tokens_to_patches", "edv_op_rowln_act", "edv_op_resblock_add", "edv_op_im2col3x3",
    "edv_op_geglu_pair", "edv_op_head_dot",
]


class EdvConfig(ctypes.Structure):
    _fields_ = [
        ("dim", ctypes.c_int32), ("depth", ctypes.c_int32), ("heads", ctypes.c_int32), ("taps", ctypes.c_int32 * 4),
        ("features", ctypes.c_int32), ("out_channels", ctypes.c_int32 * 4), ("num_frames", ctypes.c_int32),
        ("conv_head", ctypes.c_int32), ("out_sigmoid", ctypes.c_int32), ("inv_sigmoid", ctypes.c_int32),
        ("res_blocks", ctypes.c_int32), ("rope", ctypes.c_int32), ("dtype", ctypes.c_int32), ("engine", ctypes.c_int32),
        ("no_motion", ctypes.c_int32), ("no_normalize", ctypes.c_int32), ("use_clstoken", ctypes.c_int32), ("no_cls", ctypes.c_int32),
    ]


class EdvGemmDesc(ctypes.Structure):
    """Mirror of edv_gemm_desc (include/endodav_b200.h); the library rejects a struct_bytes other than its own sizeof."""
    _fields_ = [
        ("struct_bytes", ctypes.c_int32),
        ("A", ctypes.c_void_p), ("W", ctypes.c_void_p),
        ("M", ctypes.c_int32), ("N", ctypes.c_int32), ("K", ctypes.c_int32), ("lda", ctypes.c_int64),
        ("conv", ctypes.c_int32), ("F", ctypes.c_int32), ("H", ctypes.c_int32), ("Wd", ctypes.c_int32), ("C", ctypes.c_int32),
        ("stride", ctypes.c_int32),
        ("out", ctypes.c_void_p), ("out_relu", ctypes.c_void_p), ("bias", ctypes.c_void_p), ("rowbias", ctypes.c_void_p),
        ("res1", ctypes.c_void_p), ("res2", ctypes.c_void_p), ("head_w", ctypes.c_void_p),
        ("ldo", ctypes.c_int64), ("ld_res1", ctypes.c_int64), ("ld_res2", ctypes.c_int64), ("rb_ld", ctypes.c_int64),
        ("rb_div", ctypes.c_int32), ("rb_mod", ctypes.c_int32),
        ("out_f32", ctypes.c_int32), ("res1_f32", ctypes.c_int32), ("res2_f32", ctypes.c_int32),
        ("act", ctypes.c_int32), ("map", ctypes.c_int32), ("map_p", ctypes.c_int32),
        ("ps_k", ctypes.c_int32), ("ps_h", ctypes.c_int32), ("ps_w", ctypes.c_int32), ("ps_c", ctypes.c_int32),
        ("sig_sign", ctypes.c_float),
    ]


# epilogue codes of csrc/common.cuh (Epi::act, Epi::map)
ACT_NONE, ACT_GELU, ACT_RELU, ACT_GEGLU, ACT_HEAD, ACT_SIGMOID = 0, 1, 2, 3, 4, 5
MAP_LINEAR, MAP_TOKENS, MAP_PIXSHUF = 0, 1, 2


class EndoDAVError(RuntimeError):
    pass


_lib = None


def load_library():
    """Load the CUDA library; raises (never falls back) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise EndoDAVError(
            "endodav_b200: %s is missing -- build it with `python -m endodav_b200.build` "
            "(there is no CPU or PyTorch fallback for this path)" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    if not hasattr(lib, "edv_abi_version") or lib.edv_abi_version() != ABI_VERSION:
        got = lib.edv_abi_version() if hasattr(lib, "edv_abi_version") else "none"
        raise EndoDAVError("endodav_b200: %s is stale (ABI version %s, this host expects %d) -- rebuild it with "
                           "`python -m endodav_b200.build --force`" % (LIB_PATH, got, ABI_VERSION))
    vp, ci, sz = ctypes.c_void_p, ctypes.c_int, ctypes.c_size_t
    lib.edv_create.argtypes = [ctypes.POINTER(EdvConfig), ctypes.POINTER(vp)]
    lib.edv_destroy.argtypes = [vp]
    lib.edv_destroy.restype = None
    lib.edv_last_error.argtypes = [vp]
    lib.edv_last_error.restype = ctypes.c_char_p
    lib.edv_set_weight.argtypes = [vp, ctypes.c_char_p, vp, sz]
    lib.edv_plan.argtypes = [vp, ci, ci, ci, ci, ci, ci, ctypes.POINTER(sz)]
    lib.edv_forward.argtypes = [vp, vp, ctypes.POINTER(vp), vp, ci, ci, vp, vp]
    lib.edv_forward_u8.argtypes = [vp, vp, ctypes.POINTER(vp), vp, ci, ci, vp, vp]
    lib.edv_output_shape.argtypes = [vp, ci, ctypes.POINTER(ci), ctypes.POINTER(ci)]
    lib.edv_launch_count.argtypes = [vp]
    lib.edv_set_debug.argtypes = [vp, ci]
    lib.edv_debug_tap.argtypes = [vp, ctypes.c_char_p, ctypes.POINTER(sz), ctypes.POINTER(ctypes.c_longlong),
                                  ctypes.POINTER(ci)]
    lib.edv_plan_buffer.argtypes = [vp, ci, ctypes.c_char_p, ci, ctypes.POINTER(sz), ctypes.POINTER(sz), ctypes.POINTER(ci)]
    lib.edv_set_graph_mode.argtypes = [vp, ci]
    lib.edv_graph_count.argtypes = [vp]
    lib.edv_graph_status.argtypes = [vp]
    lib.edv_graph_status.restype = ctypes.c_char_p
    lib.edv_profile.argtypes = [vp, ci]
    lib.edv_profile_reset.argtypes = [vp]
    lib.edv_profile_collect.argtypes = [vp]
    lib.edv_profile_get.argtypes = [vp, ci, ctypes.c_char_p, ci, ctypes.POINTER(ctypes.c_double),
                                    ctypes.POINTER(ctypes.c_longlong), ctypes.POINTER(ctypes.c_double),
                                    ctypes.POINTER(ctypes.c_double)]
    lib.edv_op_gemm.argtypes = [ci, ci, ctypes.POINTER(EdvGemmDesc), ctypes.c_char_p, ci, vp]
    lib.edv_op_attention.argtypes = [ci, ci, vp, vp, ci, ci, ci, ctypes.c_char_p, ci, vp]
    lib.edv_op_linear_residual_ln.argtypes = [ci, vp, vp, vp, vp, vp, vp, ctypes.c_float, vp, ci, ci, ci, vp, ctypes.c_char_p, ci, vp]
    lib.edv_op_linear_timeline.argtypes = [ci, vp, vp, vp, vp, ci, ci, ci, ci, vp, vp]
    lib.edv_op_attention_timeline.argtypes = [ci, vp, vp, ci, ci, ci, vp, vp]
    lib.edv_op_temporal_attention.argtypes = [ci, vp, vp, ci, ci, ci, ci, vp, ctypes.c_char_p, ci, vp]
    lib.edv_op_disp_head.argtypes = [ci, vp, vp, vp, vp, vp, ci, ci, ci, ci, ci, ci, ctypes.c_float, ctypes.c_char_p, ci, vp]
    lib.edv_op_cubic_resize_u8.argtypes = [vp, vp, ci, ci, ci, ci, ci, vp]
    lib.edv_op_stitch_window.argtypes = [vp, ci, ci, ci, vp, vp, ci, vp, vp, vp]
    lib.edv_op_stitch_plan.argtypes = [ci, ci, vp, ctypes.c_longlong]
    lib.edv_op_disp_to_depth.argtypes = [vp, vp, vp, ctypes.c_longlong, ctypes.c_double, ctypes.c_double, vp]
    lib.edv_op_compute_errors.argtypes = [vp, vp, vp, ci, ctypes.c_longlong, ctypes.c_float, ctypes.c_float, ctypes.c_float,
                                          ctypes.c_float, ctypes.c_float, vp, vp]
    lib.edv_op_layernorm.argtypes = [ci, vp, vp, vp, vp, ci, ci, ctypes.c_float, ci, ci, vp, ci, ci, vp]
    ll, cf = ctypes.c_longlong, ctypes.c_float
    lib.edv_op_cubic_resize_u8_gather.argtypes = [vp, ci, ci, ci, ll, ll, ll, ll, vp, ci, vp, ci, ci, vp]
    lib.edv_op_preprocess_patches.argtypes = [ci, vp, ci, vp, ci, ci, ci, ci, ci, ci, vp]
    lib.edv_op_tokens_to_patches.argtypes = [ci, vp, vp, ll, ci, ci, ci, vp]
    lib.edv_op_rowln_act.argtypes = [ci, vp, vp, vp, vp, ll, ci, ci, cf, ci, vp]
    lib.edv_op_resblock_add.argtypes = [ci, vp, vp, vp, vp, ll, ci, ci, cf, ci, vp]
    lib.edv_op_im2col3x3.argtypes = [ci, vp, vp, ci, ci, ci, ci, ci, vp]
    lib.edv_op_geglu_pair.argtypes = [ci, vp, vp, ll, ci, vp]
    lib.edv_op_head_dot.argtypes = [ci, vp, vp, vp, ll, ci, cf, vp]
    lib.edv_op_groupnorm.argtypes = [ci, vp, vp, vp, vp, ci, ci, ci, ctypes.c_float, vp]
    lib.edv_op_upsample.argtypes = [ci, vp, vp, ci, ci, ci, ci, ci, ci, vp]
    lib.edv_op_resize_f32.argtypes = [vp, vp, ci, ci, ci, ci, ci, vp]
    for name in EXPORTS:
        fn = getattr(lib, name)
        if name not in ("edv_destroy", "edv_last_error", "edv_graph_status"):
            fn.restype = ci
    lib.edv_op_stitch_plan.restype = ctypes.c_longlong
    _lib = lib
    return lib


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def _check(rc, ctx=None, what=""):
    if rc != 0:
        lib = load_library()
        msg = lib.edv_last_error(ctx if ctx is not None else ctypes.c_void_p(0))
        raise EndoDAVError("%s failed (%d): %s" % (what, rc, (msg or b"").decode("utf-8", "replace")))


class Engine:
    """One ``edv_ctx``: a model on one device.  Holds the packed weights (so the borrowed device
    pointers stay alive) and one workspace per planned shape."""

    def __init__(self, cfg: EdvConfig, device):
        self.lib = load_library()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise EndoDAVError("endodav_b200 runs on CUDA devices only (got %s)" % (device,))
        self.cfg = cfg
        self.ctx = ctypes.c_void_p(0)
        with torch.cuda.device(self.device):
            _check(self.lib.edv_create(ctypes.byref(cfg), ctypes.byref(self.ctx)), None, "edv_create")
        self.weights = {}
        self.shape_key = None
        self.workspace = None
        self.debug = False

    def __del__(self):
        try:
            if getattr(self, "ctx", None) and self.ctx.value:
                self.lib.edv_destroy(self.ctx)
                self.ctx = ctypes.c_void_p(0)
        except Exception:
            pass

    def set_weights(self, packed: dict):
        for name, t in packed.items():
            t = t.to(self.device).contiguous()
            self.weights[name] = t
            _check(self.lib.edv_set_weight(self.ctx, name.encode(), _ptr(t), t.numel() * t.element_size()), self.ctx,
                   "edv_set_weight(%s)" % name)

    def set_debug(self, on: bool):
        self.debug = bool(on)
        _check(self.lib.edv_set_debug(self.ctx, int(on)), self.ctx, "edv_set_debug")
        self.shape_key = None

    def plan(self, B, T, H, W, net_h, net_w):
        key = (B, T, H, W, net_h, net_w)
        if key == self.shape_key:
            return False
        nbytes = ctypes.c_size_t(0)
        _check(self.lib.edv_plan(self.ctx, B, T, H, W, net_h, net_w, ctypes.byref(nbytes)), self.ctx, "edv_plan")
        if self.workspace is None or self.workspace.numel() < nbytes.value + 1024:
            self.workspace = None
            self.workspace = torch.empty(nbytes.value + 1024, dtype=torch.uint8, device=self.device)
        self.shape_key = key
        return True

    def _ws_ptr(self):
        base = self.workspace.data_ptr()
        return (base + 1023) & ~1023

    def output_shapes(self):
        out = []
        for s in range(4):
            h, w = ctypes.c_int(0), ctypes.c_int(0)
            _check(self.lib.edv_output_shape(self.ctx, s, ctypes.byref(h), ctypes.byref(w)), self.ctx, "edv_output_shape")
            out.append((h.value, w.value))
        return out

    def forward(self, frames, resize_to=None, want_pyramid=True, resized_out=None):
        """frames: float32 [B,T,3,H,W] (or uint8 [B*T,H,W,3] at network resolution) on this
        device.  Returns (list of 4 disparity tensors [BT,1,h_s,w_s] or None, resized or None)."""
        BT = self.shape_key[0] * self.shape_key[1]
        shapes = self.output_shapes()
        disp = [torch.empty(BT, 1, h, w, dtype=torch.float32, device=self.device) for (h, w) in shapes] if want_pyramid else None
        arr = (ctypes.c_void_p * 4)(*([_ptr(d) for d in disp] if disp else [None] * 4))
        resized = None
        oh = ow = 0
        if resize_to is not None:
            oh, ow = resize_to
            resized = resized_out if resized_out is not None else torch.empty(BT, oh, ow, dtype=torch.float32, device=self.device)
            if tuple(resized.shape) != (BT, oh, ow) or resized.dtype != torch.float32 or not resized.is_contiguous():
                raise EndoDAVError("resized_out must be a contiguous float32 [%d,%d,%d] tensor" % (BT, oh, ow))
        fn = self.lib.edv_forward_u8 if frames.dtype == torch.uint8 else self.lib.edv_forward
        rc = fn(self.ctx, _ptr(frames), arr, _ptr(resized), oh, ow, ctypes.c_void_p(self._ws_ptr()), _stream())
        _check(rc, self.ctx, "edv_forward")
        return disp, resized

    def set_graph_mode(self, on: bool):
        """CUDA-graph replay of the planned forward (default on); see include/endodav_b200.h."""
        _check(self.lib.edv_set_graph_mode(self.ctx, int(on)), self.ctx, "edv_set_graph_mode")

    def graph_count(self):
        return int(self.lib.edv_graph_count(self.ctx))

    def graph_status(self):
        return self.lib.edv_graph_status(self.ctx).decode()

    def launch_count(self):
        return int(self.lib.edv_launch_count(self.ctx))

    def profile(self, on: bool):
        """Per-launch CUDA-event timing inside edv_forward (bench.py's live roofline)."""
        _check(self.lib.edv_profile(self.ctx, int(on)), self.ctx, "edv_profile")
        if on:
            _check(self.lib.edv_profile_reset(self.ctx), self.ctx, "edv_profile_reset")

    def profile_collect(self):
        """-> list of dict(name, ms, count, flops, bytes), totals since profile(True)."""
        n = self.lib.edv_profile_collect(self.ctx)
        if n < 0:
            _check(n, self.ctx, "edv_profile_collect")
        out = []
        buf = ctypes.create_string_buffer(128)
        for i in range(n):
            ms, cnt, fl, by = ctypes.c_double(0), ctypes.c_longlong(0), ctypes.c_double(0), ctypes.c_double(0)
            _check(self.lib.edv_profile_get(self.ctx, i, buf, 128, ctypes.byref(ms), ctypes.byref(cnt), ctypes.byref(fl),
                                            ctypes.byref(by)), self.ctx, "edv_profile_get")
            out.append(dict(name=buf.value.decode(), ms=ms.value, count=cnt.value, flops=fl.value, bytes=by.value))
        return out

    def plan_buffers(self):
        """-> {name: tensor view into the workspace} for every buffer of the current plan (16-bit buffers in the
        compute dtype, float32 / float2 ones as float32).  Diagnostic: range scans of the intermediates."""
        out = {}
        buf = ctypes.create_string_buffer(64)
        base = self._ws_ptr() - self.workspace.data_ptr()
        i = 0
        while True:
            off, nb, el = ctypes.c_size_t(0), ctypes.c_size_t(0), ctypes.c_int(0)
            if self.lib.edv_plan_buffer(self.ctx, i, buf, 64, ctypes.byref(off), ctypes.byref(nb), ctypes.byref(el)) != 0:
                break
            dt = TORCH_DTYPE[self.cfg.dtype] if el.value == 2 else torch.float32
            out[buf.value.decode()] = self.workspace[base + off.value: base + off.value + nb.value].view(dt)
            i += 1
        return out

    def debug_tap(self, name):
        off, rows, cols = ctypes.c_size_t(0), ctypes.c_longlong(0), ctypes.c_int(0)
        _check(self.lib.edv_debug_tap(self.ctx, name.encode(), ctypes.byref(off), ctypes.byref(rows), ctypes.byref(cols)),
               self.ctx, "edv_debug_tap")
        start = self._ws_ptr() - self.workspace.data_ptr() + off.value
        n = rows.value * cols.value
        return self.workspace[start:start + 4 * n].view(torch.float32).view(rows.value, cols.value).clone()


# ---- thin wrappers over the per-kernel entry points (used by tests and profiling) ---------------
def _dt(t):
    return {torch.float32: EDV_F32, torch.bfloat16: EDV_BF16, torch.float16: EDV_F16}[t.dtype]


def gemm_desc(A, W, out, M=None, lda=None, conv=None, bias=None, rowbias=None, res1=None, res2=None, out_relu=None,
              head_w=None, ldo=None, ld_res1=None, ld_res2=None, rb_ld=0, rb_div=1, rb_mod=1, act=ACT_NONE, map=MAP_LINEAR,
              map_p=0, ps=(0, 0, 0, 0), sig_sign=0.0):
    """-> EdvGemmDesc for out = epilogue(A W^T).  A [M, K] (row pitch lda) or, with conv = (F, H, W, C, stride), an NHWC
    activation for a 3x3 pad-1 convolution (K = 9 C); W [N, K].  Leading dimensions default to N; ld_res1 / ld_res2 to ldo.
    out / res1 / res2 are float32 tensors (out_f32 / res*_f32) or in A's dtype; ps = (k, grid h, grid w, channels)."""
    N = W.shape[0]
    d = EdvGemmDesc()
    d.struct_bytes = ctypes.sizeof(EdvGemmDesc)
    d.A, d.W, d.N, d.K = A.data_ptr(), W.data_ptr(), N, W.shape[1]
    if conv is not None:
        d.conv = 1
        d.F, d.H, d.Wd, d.C, d.stride = conv
        d.M = M if M is not None else d.F * ((d.H - 1) // d.stride + 1) * ((d.Wd - 1) // d.stride + 1)
        d.lda = d.K
    else:
        d.M = M if M is not None else A.shape[0]
        d.lda = lda if lda is not None else A.shape[1]
        d.stride = 1
    d.out, d.out_relu = _ptr(out).value, _ptr(out_relu).value
    d.bias, d.rowbias, d.head_w = _ptr(bias).value, _ptr(rowbias).value, _ptr(head_w).value
    d.res1, d.res2 = _ptr(res1).value, _ptr(res2).value
    d.ldo = ldo if ldo is not None else N
    d.ld_res1 = ld_res1 if ld_res1 is not None else d.ldo
    d.ld_res2 = ld_res2 if ld_res2 is not None else d.ldo
    d.rb_ld, d.rb_div, d.rb_mod = rb_ld, rb_div, rb_mod
    d.out_f32 = int(out is not None and out.dtype == torch.float32)
    d.res1_f32 = int(res1 is not None and res1.dtype == torch.float32)
    d.res2_f32 = int(res2 is not None and res2.dtype == torch.float32)
    d.act, d.map, d.map_p = act, map, map_p
    d.ps_k, d.ps_h, d.ps_w, d.ps_c = ps
    d.sig_sign = sig_sign
    return d


def op_gemm_status(dtype, engine, desc):
    """-> (edv_status, name of the kernel instance that ran, e.g. "gemm_tc<BN=32,BK=64,kind=0x9,tma=0>")."""
    lib = load_library()
    name = ctypes.create_string_buffer(128)
    # without a device there is no stream; the library then rejects the call or fails at the launch
    stream = _stream() if torch.cuda.is_available() else ctypes.c_void_p(0)
    rc = lib.edv_op_gemm(dtype, engine, ctypes.byref(desc), name, 128, stream)
    return rc, name.value.decode()


def op_gemm(A, W, out, engine=ENGINE_TC, **epi):
    """out (and epi["out_relu"]) = the fused epilogue of A W^T (gemm_desc), through the forward's own GEMM dispatcher;
    returns the kernel instance that ran."""
    rc, kernel = op_gemm_status(_dt(A), engine, gemm_desc(A, W, out, **epi))
    _check(rc, None, "edv_op_gemm")
    return kernel


def op_linear(A, W, bias=None, act=0, engine=ENGINE_TC):
    M = A.shape[0]
    C = torch.empty(M, W.shape[0], dtype=A.dtype, device=A.device)
    op_gemm(A, W, C, engine, bias=bias, act=act)
    return C


def op_linear_residual_ln_kernel(A, W, bias, x, gamma=None, beta=None, eps=1e-6, xn=None, timeline=None):
    """-> (xn, name of the kernel instance that ran, e.g. "gemm_ln<bf16>").  x (float32 [M,384], updated IN PLACE) +=
    A W^T + bias; xn = LayerNorm(x) in A's dtype, None without gamma.  xn: optional caller-owned buffer whose first M rows
    receive it.  timeline: optional int64 [64] device tensor receiving the kernel's own epilogue time stamps."""
    lib = load_library()
    M, K = A.shape
    N = W.shape[0]
    if gamma is not None and xn is None:
        xn = torch.empty(M, N, dtype=A.dtype, device=A.device)
    name = ctypes.create_string_buffer(128)
    _check(lib.edv_op_linear_residual_ln(_dt(A), _ptr(A), _ptr(W), _ptr(bias), _ptr(x), _ptr(gamma), _ptr(beta), ctypes.c_float(eps),
                                         _ptr(xn), M, N, K, _ptr(timeline), name, 128, _stream()), None, "edv_op_linear_residual_ln")
    return xn, name.value.decode()


def op_linear_residual_ln(A, W, bias, x, gamma=None, beta=None, eps=1e-6, timeline=None):
    """x (float32 [M,384], updated IN PLACE) += A W^T + bias; returns LayerNorm(x) in A's dtype (None without gamma).
    timeline: optional int64 [64] device tensor receiving the kernel's own epilogue time stamps."""
    return op_linear_residual_ln_kernel(A, W, bias, x, gamma, beta, eps, timeline=timeline)[0]


def op_linear_timeline(A, W, bias=None, act=0):
    """-> (C, int64 [4,256] clock64 stamps of the first 4 CTAs); slot table in csrc/gemm_tc.cuh."""
    lib = load_library()
    M, K = A.shape
    N = W.shape[0]
    C = torch.empty(M, N, dtype=A.dtype, device=A.device)
    tl = torch.zeros(4, 256, dtype=torch.int64, device=A.device)
    _check(lib.edv_op_linear_timeline(_dt(A), _ptr(A), _ptr(W), _ptr(bias), _ptr(C), M, N, K, act, _ptr(tl), _stream()), None,
           "edv_op_linear_timeline")
    return C, tl


def op_conv3x3(X, Wt, bias=None, relu_out=False, engine=ENGINE_TC):
    F, H, W, Cin = X.shape
    Y = torch.empty(F, H, W, Wt.shape[0], dtype=X.dtype, device=X.device)
    op_gemm(X, Wt, Y, engine, conv=(F, H, W, Cin, 1), bias=bias, act=ACT_RELU if relu_out else ACT_NONE)
    return Y


def op_attention_kernel(qkv, F, S, heads, engine=ENGINE_TC, out=None):
    """-> (out [F*S, heads*64], name of the kernel instance that ran, e.g. "flash_attention_tc<bf16>").  out: optional
    caller-owned buffer whose first F*S rows receive the result."""
    lib = load_library()
    if out is None:
        out = torch.empty(F * S, heads * 64, dtype=qkv.dtype, device=qkv.device)
    name = ctypes.create_string_buffer(128)
    _check(lib.edv_op_attention(_dt(qkv), engine, _ptr(qkv), _ptr(out), F, S, heads, name, 128, _stream()), None,
           "edv_op_attention")
    return out, name.value.decode()


def op_attention(qkv, F, S, heads, engine=ENGINE_TC):
    return op_attention_kernel(qkv, F, S, heads, engine)[0]


def op_attention_timeline(qkv, F, S, heads):
    """-> (out, int64 [8,64] clock64 stamps of the first 8 CTAs); slot table in csrc/attention_tc.cuh."""
    lib = load_library()
    out = torch.empty(F * S, heads * 64, dtype=qkv.dtype, device=qkv.device)
    tl = torch.zeros(8, 64, dtype=torch.int64, device=qkv.device)
    _check(lib.edv_op_attention_timeline(_dt(qkv), _ptr(qkv), _ptr(out), F, S, heads, _ptr(tl), _stream()), None,
           "edv_op_attention_timeline")
    return out, tl


def op_temporal_attention_kernel(qkv, B, T, hw, C, rope=None, out=None):
    """-> (out [B*T*hw, C], name of the kernel instance that ran).  rope: float32 [T, C] = [T][C/2] (cos, sin) pairs
    (pack.py), or None."""
    lib = load_library()
    if out is None:
        out = torch.empty(B * T * hw, C, dtype=qkv.dtype, device=qkv.device)
    name = ctypes.create_string_buffer(128)
    _check(lib.edv_op_temporal_attention(_dt(qkv), _ptr(qkv), _ptr(out), B, T, hw, C, _ptr(rope), name, 128, _stream()), None,
           "edv_op_temporal_attention")
    return out, name.value.decode()


def op_temporal_attention(qkv, B, T, hw, C, rope=None):
    return op_temporal_attention_kernel(qkv, B, T, hw, C, rope)[0]


def op_disp_head_kernel(X, Wt, bias, head_w, oh, ow, sig_sign=0.0, out=None):
    """-> (out [F, oh, ow] float32, name of the kernel instance that ran, e.g. "head_fused<bf16,CIN=128>").  X: NHWC
    [F, H1, W1, Cin]; out: optional caller-owned float32 buffer whose first F*oh*ow elements receive the result."""
    lib = load_library()
    F, H1, W1, Cin = X.shape
    if out is None:
        out = torch.empty(F, oh, ow, dtype=torch.float32, device=X.device)
    name = ctypes.create_string_buffer(128)
    _check(lib.edv_op_disp_head(_dt(X), _ptr(X), _ptr(Wt), _ptr(bias), _ptr(head_w), _ptr(out), F, H1, W1, oh, ow, Cin,
                                ctypes.c_float(sig_sign), name, 128, _stream()), None, "edv_op_disp_head")
    return out, name.value.decode()


def op_disp_head(X, Wt, bias, head_w, oh, ow, sig_sign=0.0):
    return op_disp_head_kernel(X, Wt, bias, head_w, oh, ow, sig_sign)[0]


def op_cubic_resize_u8(frames_u8, h, w, out=None, index=None):
    """uint8 [n_src,H,W,3] (device, any positive strides; a size-1 dimension may have any stride) -> float32 [N,3,h,w]: the reference's per-frame cv2 cubic resize of
    frame/255.  index: the source frame of every output frame (N = len(index)); default every frame in order."""
    import numpy as np

    lib = load_library()
    if frames_u8.dtype != torch.uint8 or frames_u8.dim() != 4 or frames_u8.shape[3] != 3:
        raise EndoDAVError("op_cubic_resize_u8: frames must be a uint8 [N,H,W,3] tensor, got %s %s"
                           % (frames_u8.dtype, tuple(frames_u8.shape)))
    n_src, H, W, _ = frames_u8.shape
    if index is not None:
        index = np.ascontiguousarray(index, dtype=np.int64).reshape(-1)
    N = n_src if index is None else index.size
    if out is None:
        out = torch.empty(N, 3, h, w, dtype=torch.float32, device=frames_u8.device)
    elif tuple(out.shape) != (N, 3, h, w) or out.dtype != torch.float32 or not out.is_contiguous():
        raise EndoDAVError("op_cubic_resize_u8: out must be a contiguous float32 [%d,3,%d,%d] tensor" % (N, h, w))
    if index is None and frames_u8.is_contiguous():
        _check(lib.edv_op_cubic_resize_u8(_ptr(frames_u8), _ptr(out), N, H, W, h, w, _stream()), None, "edv_op_cubic_resize_u8")
        return out
    if index is None:
        index = np.arange(n_src, dtype=np.int64)
    # the stride of a size-1 dimension is never used; torch may report any value for it
    strides = [s if d > 1 else 1 for s, d in zip(frames_u8.stride(), frames_u8.shape)]
    _check(lib.edv_op_cubic_resize_u8_gather(_ptr(frames_u8), n_src, H, W, *strides, index.ctypes.data_as(ctypes.c_void_p), N,
                                             _ptr(out), h, w, _stream()), None, "edv_op_cubic_resize_u8_gather")
    return out


def op_layernorm(X, gamma, beta, eps, out_dtype, grp=0, skip=0, add=None, add_div=1, add_mod=1, out=None):
    """LayerNorm of the rows of X (float32 [rows, D]) into out_dtype, with the row selection grp / skip and the additive
    per-frame table add of edv_op_layernorm.  out: optional [>= M, D] buffer (its first M rows are written)."""
    lib = load_library()
    rows, D = X.shape
    M = rows if grp == 0 else (rows // grp) * (grp - skip if skip >= 0 else -skip)
    Y = out if out is not None else torch.empty(M, D, dtype=out_dtype, device=X.device)
    _check(lib.edv_op_layernorm(_dt(Y), _ptr(X), _ptr(gamma), _ptr(beta), _ptr(Y), M, D, ctypes.c_float(eps), grp, skip, _ptr(add),
                                add_div, add_mod, _stream()), None, "edv_op_layernorm")
    return Y


def op_preprocess_patches(frames, h, w, out, normalize=True):
    """frames float32 [F,3,H,W] or uint8 [F,H,W,3] (at h x w) -> out [F*(h/14)*(w/14), 640] (out's dtype)."""
    lib = load_library()
    u8 = frames.dtype == torch.uint8
    Fr, H, W = (frames.shape[0], frames.shape[1], frames.shape[2]) if u8 else (frames.shape[0], frames.shape[2], frames.shape[3])
    _check(lib.edv_op_preprocess_patches(_dt(out), _ptr(frames), int(u8), _ptr(out), Fr, H, W, h, w, int(normalize), _stream()), None,
           "edv_op_preprocess_patches")
    return out


def op_tokens_to_patches(x, out, Mp, P, D, cls):
    """out [Mp, D] (out's dtype) = the patch rows of the float32 token stream x [Mp/P, P + cls, D]."""
    lib = load_library()
    _check(lib.edv_op_tokens_to_patches(_dt(out), _ptr(x), _ptr(out), Mp, P, D, cls, _stream()), None, "edv_op_tokens_to_patches")
    return out


def op_rowln_act(x, gamma, beta, y, M, C, Cr, eps=1e-6, gelu=True):
    """y [M, C] = GELU(LayerNorm over the first Cr channels of x [M, C]), padding columns 0 (x's dtype)."""
    lib = load_library()
    _check(lib.edv_op_rowln_act(_dt(x), _ptr(x), _ptr(gamma), _ptr(beta), _ptr(y), M, C, Cr, ctypes.c_float(eps), int(gelu), _stream()),
           None, "edv_op_rowln_act")
    return y


def op_resblock_add(x, r, gamma, beta, Mp, P, D, cls, eps=1e-6):
    """x (float32 token stream, in place): patch rows += LayerNorm(r [Mp, D]) (r's dtype)."""
    lib = load_library()
    _check(lib.edv_op_resblock_add(_dt(r), _ptr(x), _ptr(r), _ptr(gamma), _ptr(beta), Mp, P, D, ctypes.c_float(eps), cls, _stream()),
           None, "edv_op_resblock_add")
    return x


def op_im2col3x3(x, out, stride=2):
    """NHWC x [F,H,W,C] -> out [F*OH*OW, 9*C] (3x3, pad 1, (ky,kx,c) order)."""
    lib = load_library()
    Fr, H, W, C = x.shape
    _check(lib.edv_op_im2col3x3(_dt(x), _ptr(x), _ptr(out), Fr, H, W, C, stride, _stream()), None, "edv_op_im2col3x3")
    return out


def op_geglu_pair(hg, out, M, C4):
    """out [M, C4] = value * gelu(gate) of hg [M, 2*C4] in [64 value | 64 gate] column blocks (hg's dtype)."""
    lib = load_library()
    _check(lib.edv_op_geglu_pair(_dt(hg), _ptr(hg), _ptr(out), M, C4, _stream()), None, "edv_op_geglu_pair")
    return out


def op_head_dot(x, w, out, M, C, sig_sign=0.0):
    """out [M] float32 = x [M, C] . w[:C] + w[C], then ReLU (sig_sign 0) or sigmoid(sig_sign * .)."""
    lib = load_library()
    _check(lib.edv_op_head_dot(_dt(x), _ptr(x), _ptr(w), _ptr(out), M, C, ctypes.c_float(sig_sign), _stream()), None, "edv_op_head_dot")
    return out


def op_groupnorm(X, gamma, beta, eps):
    lib = load_library()
    F, hw, C = X.shape
    Y = torch.empty_like(X)
    _check(lib.edv_op_groupnorm(_dt(X), _ptr(X), _ptr(gamma), _ptr(beta), _ptr(Y), F, hw, C, ctypes.c_float(eps), _stream()), None,
           "edv_op_groupnorm")
    return Y


def op_upsample(X, oh, ow):
    lib = load_library()
    F, h, w, C = X.shape
    Y = torch.empty(F, oh, ow, C, dtype=X.dtype, device=X.device)
    _check(lib.edv_op_upsample(_dt(X), _ptr(X), _ptr(Y), F, h, w, oh, ow, C, _stream()), None, "edv_op_upsample")
    return Y


def op_resize_f32(X, oh, ow):
    lib = load_library()
    F, h, w = X.shape
    Y = torch.empty(F, oh, ow, dtype=torch.float32, device=X.device)
    _check(lib.edv_op_resize_f32(_ptr(X), _ptr(Y), F, h, w, oh, ow, _stream()), None, "edv_op_resize_f32")
    return Y


def stitch_plan(H, W):
    """numpy's pairwise-summation tree for the 8*H*W overlap elements as an int32 table (host only, no GPU
    needed): [L, I, levels, root, level starts..., L+1 leaf offsets, I (left,right) pairs]."""
    import numpy as np

    lib = load_library()
    need = lib.edv_op_stitch_plan(H, W, None, 0)
    if need < 0:
        raise EndoDAVError("edv_op_stitch_plan(%d,%d) failed (%d): overlap of 8*H*W elements must stay below 2^24" % (H, W, need))
    plan = np.empty(need, dtype=np.int32)
    got = lib.edv_op_stitch_plan(H, W, plan.ctypes.data_as(ctypes.c_void_p), need)
    assert got == need
    return plan


def op_stitch_window(win, k, out, plan_dev, n_leaves, scratch, scale_shift, base_frame=0):
    """Append window k ([32,H,W] float32, device) to the stitched sequence on the current stream: the reference's
    scale/shift alignment + cross-fade (endodav.py:213-254), no host sync.  ``out[i]`` holds frame
    ``base_frame + i`` of the sequence (base_frame = 0: ``out`` is the whole [32+22*(nwin-1),H,W] sequence); window k
    touches frames [10+22k-8, 10+22k+22), which must lie inside ``out``."""
    lib = load_library()
    _, H, W = win.shape
    lo = 0 if k == 0 else 10 + 22 * k - 8
    hi = 32 if k == 0 else 10 + 22 * k + 22
    if lo < base_frame or hi - base_frame > out.shape[0]:
        raise EndoDAVError("op_stitch_window: window %d touches frames [%d,%d) outside the buffer [%d,%d)"
                           % (k, lo, hi, base_frame, base_frame + out.shape[0]))
    out_ptr = ctypes.c_void_p(out.data_ptr() - base_frame * H * W * 4)
    _check(lib.edv_op_stitch_window(_ptr(win), int(k), H, W, out_ptr, _ptr(plan_dev), int(n_leaves), _ptr(scratch),
                                    _ptr(scale_shift), _stream()), None, "edv_op_stitch_window")
