// endodav_b200 engine: context, weight registry, shape plan and the forward graph of
// endodav.forward (models/endodav/endodav.py:150-160) expressed as a fixed sequence of
// sm_100a kernel launches on the caller's stream.  C ABI in include/endodav_b200.h.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <map>
#include <string>
#include <unordered_map>
#include <vector>

#include "ops.cuh"
#include "stitch.cuh"
#include "metrics.cuh"

using namespace edv;

namespace {

std::string g_create_error;

struct WeightRef {
  const void* ptr;
  size_t bytes;
};

struct Buf {
  size_t off = 0;
  size_t bytes = 0;
  int elem = 0;   // element size in bytes (4: float32 regardless of the activation dtype; 8: float2 statistics)
};

struct DebugTap {
  Buf buf;            // float32 snapshot
  long long rows = 0;
  int cols = 0;
};

struct MMPlan {
  int C = 0, h = 0, w = 0;
};

struct Plan {
  bool valid = false;
  int B = 0, T = 0, H = 0, W = 0, h = 0, w = 0;
  int BT = 0, ph = 0, pw = 0, P = 0, N = 0;
  long long M = 0, Mp = 0;
  int ph2 = 0, pw2 = 0;
  int Cp[4] = {0, 0, 0, 0};
  int out_h[4] = {0, 0, 0, 0}, out_w[4] = {0, 0, 0, 0};
  MMPlan mm[4];
  size_t total = 0;
  std::map<std::string, Buf> bufs;
  std::map<std::string, DebugTap> taps;
};

inline int round_up(int v, int m) { return (v + m - 1) / m * m; }

}  // namespace

// One captured forward: the launch sequence of Fwd::run for one planned shape and one set of external INPUT /
// workspace pointers.  The disparity pyramid is written into the plan's own buffers inside the graph and copied to the
// caller's tensors behind the replay (copy_pyramid_out, ~20 us at 32 x 518 x 518): callers get fresh output tensors from
// their allocator on every call, and a key that included them made the end-to-end loop capture or run eagerly again and
// again (measured: e2e anywhere between 75 % and 100 % of the device-timed rate).  One set of
// pointers (the kernel arguments -- including the tensor maps, which are __grid_constant__ parameters -- are
// baked into the graph's kernel nodes, so nothing is encoded or launched from the host when it is replayed).
struct GraphEntry {
  const void* frames = nullptr;
  const void* resized = nullptr;
  const void* workspace = nullptr;
  int u8 = 0, out_h = 0, out_w = 0;
  cudaGraphExec_t exec = nullptr;
  int launches = 0;
  unsigned long long last_use = 0;
  bool same(const GraphEntry& o) const {
    return frames == o.frames && resized == o.resized && workspace == o.workspace && u8 == o.u8 && out_h == o.out_h && out_w == o.out_w;
  }
};

struct edv_ctx {
  edv_config cfg;
  std::unordered_map<std::string, WeightRef> weights;
  Plan plan;
  std::string err;
  int last_launches = 0;
  int debug = 0;
  int Kp = 640;
  // CUDA-graph replay of the planned forward (EDV_GRAPH=0 disables): up to GRAPH_SLOTS pointer sets per plan
  static constexpr int GRAPH_SLOTS = 32;
  int graph_mode = 1;
  bool plan_warm = false;              // the first forward of a plan runs eagerly (one-time cudaFuncSetAttribute etc.)
  unsigned long long graph_clock = 0;
  std::vector<GraphEntry> graphs;
  std::vector<GraphEntry> seen;        // pointer sets met once (no graph yet): a set is captured the SECOND time it comes by
  // Independent decoder branches (the three shallow reassemble paths + their temporal module) run on a low-priority
  // side stream, forked / joined with events, beside the deep path that is the critical chain (EDV_BRANCH=0: serial)
  int branch_mode = 1;
  cudaStream_t side_stream = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  bool ensure_side() {
    if (side_stream) return true;
    int lo = 0, hi = 0;
    cudaDeviceGetStreamPriorityRange(&lo, &hi);
    if (cudaStreamCreateWithPriority(&side_stream, cudaStreamNonBlocking, lo) != cudaSuccess ||
        cudaEventCreateWithFlags(&ev_fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&ev_join, cudaEventDisableTiming) != cudaSuccess) {
      cudaGetLastError();
      branch_mode = 0;
      return false;
    }
    return true;
  }
  cudaStream_t cap_stream = nullptr;   // private capture stream: the caller's stream may be the legacy default stream, which cannot be captured
  std::string graph_note = "no capture attempted";   // why the last capture attempt did not produce a graph (edv_graph_status)
  void drop_graphs() {
    for (GraphEntry& g : graphs)
      if (g.exec) cudaGraphExecDestroy(g.exec);
    graphs.clear();
    seen.clear();
    plan_warm = false;
  }
  ~edv_ctx() {
    drop_graphs();
    if (cap_stream) cudaStreamDestroy(cap_stream);
    if (side_stream) cudaStreamDestroy(side_stream);
    if (ev_fork) cudaEventDestroy(ev_fork);
    if (ev_join) cudaEventDestroy(ev_join);
  }
  Profiler prof;
  struct Agg {
    double ms = 0, flops = 0, bytes = 0;
    long long count = 0;
  };
  std::map<std::string, Agg> prof_agg;
  std::vector<std::string> prof_names;  // stable order for edv_profile_get
};

namespace {

const int KPATCH = 640;  // 3*14*14 = 588 padded to a multiple of 64

struct Fwd {
  edv_ctx* c;
  Launch L;
  unsigned char* ws;
  int dt, eng;
  size_t es;  // element size of the activation dtype
  cudaStream_t main_s;
  bool par;   // fork the independent decoder branches onto ctx->side_stream (never while profiling / tapping: both assume one serial stream)

  Fwd(edv_ctx* ctx, void* workspace, cudaStream_t s) : c(ctx), ws((unsigned char*)workspace), main_s(s) {
    L.stream = s;
    L.prof = &ctx->prof;
    dt = ctx->cfg.dtype;
    eng = ctx->cfg.dtype == EDV_F32 ? EDV_ENGINE_SIMT : ctx->cfg.engine;
    es = dtype_size(dt);
    par = ctx->branch_mode && !ctx->prof.on && !ctx->debug && ctx->ensure_side();
  }
  // fork: the side stream starts after everything launched on the main stream so far; join: the main stream waits for it
  void fork_side() {
    if (!par || !L.ok()) return;
    if (cudaEventRecord(c->ev_fork, main_s) != cudaSuccess || cudaStreamWaitEvent(c->side_stream, c->ev_fork, 0) != cudaSuccess)
      return L.fail(EDV_ERR_CUDA, std::string("fork onto the side stream: ") + cudaGetErrorString(cudaGetLastError()));
    L.stream = c->side_stream;
  }
  void back_to_main() { L.stream = main_s; }
  void join_side() {
    if (!par) return;
    L.stream = main_s;
    if (cudaEventRecord(c->ev_join, c->side_stream) != cudaSuccess || cudaStreamWaitEvent(main_s, c->ev_join, 0) != cudaSuccess)
      L.fail(EDV_ERR_CUDA, std::string("join of the side stream: ") + cudaGetErrorString(cudaGetLastError()));
  }
  bool tc() const { return eng == EDV_ENGINE_TC; }

  void* buf(const char* name) {
    auto it = c->plan.bufs.find(name);
    if (it == c->plan.bufs.end()) {
      L.fail(EDV_ERR_STATE, std::string("internal: unknown buffer ") + name);
      return ws;
    }
    return ws + it->second.off;
  }
  const void* w(const std::string& name, size_t min_bytes = 0) {
    auto it = c->weights.find(name);
    if (it == c->weights.end()) {
      L.fail(EDV_ERR_WEIGHT, "missing packed weight '" + name + "'");
      return nullptr;
    }
    if (min_bytes && it->second.bytes < min_bytes) {
      char b[64];
      snprintf(b, sizeof b, " (%zu < %zu bytes)", it->second.bytes, min_bytes);
      L.fail(EDV_ERR_WEIGHT, "packed weight '" + name + "' too small" + b);
      return nullptr;
    }
    return it->second.ptr;
  }
  const float* wf(const std::string& name, size_t n) { return (const float*)w(name, n * 4); }
  const void* wt(const std::string& name, size_t n) { return w(name, n * es); }

  // call-site tag for the profiler: the packed weight name without its indices
  // ("blk3.fc1.w" -> "blk.fc1", "ref1.rcu2.c1.w" -> "ref.rcu.c1")
  static std::string tag_of(const std::string& wname) {
    std::string t = wname;
    if (t.size() > 2 && t.compare(t.size() - 2, 2, ".w") == 0) t.resize(t.size() - 2);
    std::string o;
    for (size_t i = 0; i < t.size(); ++i) {
      const bool digit = t[i] >= '0' && t[i] <= '9';
      if (digit) {
        size_t j = i;
        while (j < t.size() && t[j] >= '0' && t[j] <= '9') ++j;
        if (j < t.size() && t[j] == '.') { i = j - 1; continue; }   // an index token: drop it
      }
      o.push_back(t[i]);
    }
    return o;
  }

  // ---- building blocks --------------------------------------------------------------------
  void linear(const void* A, long long M, int K, const std::string& wname, int N, Epi e) {
    GemmArgs a;
    a.A = A; a.W = wt(wname, (size_t)N * K); a.M = (int)M; a.N = N; a.K = K; a.lda = K; a.e = e;
    if (!L.ok()) return;
    L.tag = tag_of(wname);
    gemm(L, dt, eng, a);
    L.tag.clear();
  }
  void conv3(const void* X, int F, int H, int Wd, int C, const std::string& wname, int N, Epi e) {
    GemmArgs a;
    a.A = X; a.W = wt(wname, (size_t)N * 9 * C); a.M = F * H * Wd; a.N = N; a.K = 9 * C; a.e = e;
    a.conv = true; a.F = F; a.H = H; a.Wd = Wd; a.C = C; a.stride = 1;
    if (!L.ok()) return;
    L.tag = tag_of(wname);
    gemm(L, dt, eng, a);
    L.tag.clear();
  }
  Epi ep(void* out, long long ldo, const float* bias) {
    Epi e = epi_zero();
    e.out = out; e.ldo = ldo; e.bias = bias;
    return e;
  }
  void snapshot(const char* name, const void* src, bool src_f32, long long rows, int cols_src, int cols) {
    if (!c->debug || !L.ok()) return;
    auto it = c->plan.taps.find(name);
    if (it == c->plan.taps.end()) return;
    float* dst = (float*)(ws + it->second.buf.off);
    long long n = rows * cols;
    if (src_f32) copy_channels_f32_kernel<float><<<nblk(n, 256), 256, 0, L.stream>>>((const float*)src, dst, rows, cols_src, cols);
    else EDV_DISPATCH_T(dt, { copy_channels_f32_kernel<T><<<nblk(n, 256), 256, 0, L.stream>>>((const T*)src, dst, rows, cols_src, cols); });
    L.check("debug snapshot");
  }

  // TemporalModule (motion_module.py:60-65,102-126,164-177): X [BT*hw, C] NHWC -> Y same
  // `set`: scratch buffer family ("mm." on the main stream, "mmb." for the module that runs beside it on the side stream)
  void motion(int j, const void* X, void* Y, const std::string& set = "mm.") {
    const Plan& p = c->plan;
    const int C = p.mm[j].C, hw = p.mm[j].h * p.mm[j].w, T = p.T, B = p.B;
    const long long Mm = (long long)p.BT * hw;
    const std::string n = "mm" + std::to_string(j) + ".";
    void* gnb = buf((set + "gn").c_str());
    float* hs = (float*)buf((set + "hs").c_str());
    void* lnb = buf((set + "ln").c_str());
    void* qkvb = buf((set + "qkv").c_str());
    void* att = buf((set + "att").c_str());
    void* gg = buf((set + "gg").c_str());
    void* hsT = buf((set + "hsT").c_str());
    groupnorm(L, dt, X, wf(n + "gn.w", C), wf(n + "gn.b", C), gnb, (float2*)buf((set + "stats").c_str()), p.BT, hw, C, 1e-6f);
    {
      Epi e = ep(hs, C, wf(n + "pin.b", C));
      e.out_f32 = 1;
      linear(gnb, Mm, C, n + "pin.w", C, e);
    }
    for (int a = 0; a < 2; ++a) {
      const std::string an = n + "a" + std::to_string(a) + ".";
      // LN, + sinusoidal PE of the row's frame (motion_module.py:236-237), then q|k|v in one GEMM
      layernorm(L, dt, hs, wf(an + "ln.w", C), wf(an + "ln.b", C), lnb, Mm, C, 1e-5f, 0, 0,
                c->cfg.rope ? nullptr : wf(an + "pe", (size_t)T * C), hw, T);
      linear(lnb, Mm, C, an + "qkv.w", 3 * C, ep(qkvb, 3 * C, nullptr));
      temporal_attention(L, dt, qkvb, att, B, T, hw, C, c->cfg.rope ? wf(an + "rope", (size_t)T * C) : nullptr);
      {
        Epi e = ep(hs, C, wf(an + "out.b", C));
        e.out_f32 = 1; e.res1 = hs; e.res1_f32 = 1; e.ld_res1 = C;
        linear(att, Mm, C, an + "out.w", C, e);
      }
    }
    layernorm(L, dt, hs, wf(n + "ffln.w", C), wf(n + "ffln.b", C), lnb, Mm, C, 1e-5f);
    if (tc()) {
      Epi e = ep(gg, 4 * C, wf(n + "geglu.b", 8 * C));
      e.act = ACT_GEGLU;
      linear(lnb, Mm, C, n + "geglu.w", 8 * C, e);
    } else {
      void* tmp = buf((set + "gg2").c_str());
      linear(lnb, Mm, C, n + "geglu.w", 8 * C, ep(tmp, 8 * C, wf(n + "geglu.b", 8 * C)));
      if (L.ok()) {
        long long tot = Mm * 4 * C;
        EDV_DISPATCH_T(dt, { geglu_pair_kernel<T><<<nblk(tot, 256), 256, 0, L.stream>>>((const T*)tmp, (T*)gg, Mm, 4 * C); });
        L.check("geglu");
      }
    }
    {
      Epi e = ep(hsT, C, wf(n + "ff2.b", C));
      e.res1 = hs; e.res1_f32 = 1; e.ld_res1 = C;
      linear(gg, Mm, 4 * C, n + "ff2.w", C, e);
    }
    {
      Epi e = ep(Y, C, wf(n + "pout.b", C));
      e.res1 = X; e.ld_res1 = C;
      linear(hsT, Mm, C, n + "pout.w", C, e);
    }
  }

  // ResidualConvUnit (util/blocks.py:78-91): out = conv2(relu(conv1(relu(x)))) + x (+ extra)
  //   xr = relu(x) (written by x's producer), out_relu optionally receives relu(out)
  void rcu(const std::string& n, const void* x, const void* xr, const void* extra, void* out, void* out_relu, int F_,
           int H, int Wd, int C, void* tmp) {
    Epi e1 = ep(tmp, C, wf(n + "c1.b", C));
    e1.act = ACT_RELU;
    conv3(xr, F_, H, Wd, C, n + "c1.w", C, e1);
    Epi e2 = ep(out, C, wf(n + "c2.b", C));
    e2.res1 = x; e2.ld_res1 = C;
    if (extra) { e2.res2 = extra; e2.ld_res2 = C; }
    e2.out_relu = out_relu;
    conv3(tmp, F_, H, Wd, C, n + "c2.w", C, e2);
  }

  // FeatureFusionBlock (util/blocks.py:134-162).  out_conv (1x1, linear) commutes with the
  // bilinear resize, so it runs at the low resolution first (4x fewer FLOPs).
  //   x0 : main input (raw); x0r = relu(x0) needed only when x1 == nullptr
  //   x1 / x1r : skip input and its relu copy (nullable)
  void fusion(int k, const void* x0, const void* x0r, const void* x1, const void* x1r, int H, int Wd, int OH, int OW,
              void* out) {
    const Plan& p = c->plan;
    const int C = c->cfg.features;
    const std::string n = "ref" + std::to_string(k) + ".";
    void* tmp = buf("ref.tmp");
    void* s = buf("ref.s");
    void* sr = buf("ref.sr");
    void* u = buf("ref.u");
    void* v = buf("ref.v");
    const void* in = x0;
    const void* inr = x0r;
    if (x1) {
      rcu(n + "rcu1.", x1, x1r, x0, s, sr, p.BT, H, Wd, C, tmp);  // s = x0 + RCU1(x1)
      in = s;
      inr = sr;
    }
    rcu(n + "rcu2.", in, inr, nullptr, u, nullptr, p.BT, H, Wd, C, tmp);
    linear(u, (long long)p.BT * H * Wd, C, n + "out.w", C, ep(v, C, wf(n + "out.b", C)));
    upsample(L, dt, v, out, p.BT, H, Wd, OH, OW, C);
  }

  // disparity head on a feature map X [BT,H,W,F]: conv3x3 F->F/2, bilinear to (OH,OW),
  // conv3x3 F/2->32 + ReLU, 1x1 -> 1, then ReLU (output_conv2, dpt.py:117-124) or
  // sigmoid(sign*x) (HeadDepth, layers.py:206-217 + dpt_pyramid.py:104-109).
  void disp_head(const std::string& c0, const std::string& c2, const std::string& c4, const void* X, int H, int Wd,
                 int OH, int OW, float sig_sign, float* out) {
    const Plan& p = c->plan;
    const int F_ = c->cfg.features, Fh = F_ / 2;
    void* o1 = buf("head.o1");
    conv3(X, p.BT, H, Wd, F_, c0 + ".w", Fh, ep(o1, Fh, wf(c0 + ".b", Fh)));
    const float* hw_ = wf(c4 + ".w", 33);
    if (tc() && head_fused_supported(dt, Fh)) {
      // K14: the upsampled map and the 32-channel conv output never touch HBM
      L.tag = tag_of(c2);
      head_fused(L, dt, o1, wt(c2 + ".w", (size_t)32 * 9 * Fh), wf(c2 + ".b", 32), hw_, out, p.BT, H, Wd, OH, OW, Fh, sig_sign);
      L.tag.clear();
      return;
    }
    void* up = buf("head.up");
    upsample(L, dt, o1, up, p.BT, H, Wd, OH, OW, Fh);
    if (tc()) {
      Epi e = ep(out, 1, wf(c2 + ".b", 32));
      e.act = ACT_HEAD; e.head_w = hw_; e.sig_sign = sig_sign; e.out_f32 = 1;
      e.head_b = 0.f;  // the kernel adds head_w[32]
      conv3(up, p.BT, OH, OW, Fh, c2 + ".w", 32, e);
    } else {
      void* t32 = buf("head.t32");
      Epi e = ep(t32, 32, wf(c2 + ".b", 32));
      e.act = ACT_RELU;
      conv3(up, p.BT, OH, OW, Fh, c2 + ".w", 32, e);
      if (L.ok()) {
        long long Mh = (long long)p.BT * OH * OW;
        EDV_DISPATCH_T(dt, {
          head_dot_kernel<T><<<nblk(Mh, 256), 256, 0, L.stream>>>((const T*)t32, hw_, out, Mh, 32, sig_sign == 0.f, sig_sign,
                                                                sig_sign != 0.f);
        });
        L.check("head_dot");
      }
    }
  }

  int run(const void* frames, bool u8, float* const disp[4], float* resized, int out_h, int out_w) {
    const Plan& p = c->plan;
    const edv_config& g = c->cfg;
    const int D = g.dim;
    L.begin();
    // ---- K1 + K2: preprocess, patch embedding (patch_embed.py:75-77; vision_transformer.py:219-227)
    void* A0 = buf("A0");
    float* x = (float*)buf("x");
    {
      long long tot = p.Mp * KPATCH;
      unsigned blocks = nblk(tot / 8, 256);
      L.note(0, (double)p.BT * 3 * p.H * p.W * (u8 ? 1 : 4) + (double)tot * es);
      EDV_DISPATCH_T(dt, {
        const int nrm = g.no_normalize ? 0 : 1;  // endodac with pre_norm=False feeds raw [0,1] pixels (endodac.py:208-211)
        if (u8) preprocess_patches_kernel<T, true><<<blocks, 256, 0, L.stream>>>(frames, (T*)A0, p.BT, p.H, p.W, p.h, p.w, KPATCH, nrm);
        else preprocess_patches_kernel<T, false><<<blocks, 256, 0, L.stream>>>(frames, (T*)A0, p.BT, p.H, p.W, p.h, p.w, KPATCH, nrm);
      });
      L.check("preprocess");
      const float* cls = g.no_cls ? nullptr : wf("cls_row", D);
      if (cls && L.ok()) {
        edv::launch_k(cls_row_kernel, dim3(nblk((long long)p.BT * D, 256)), dim3(256), 0, L.stream, x, cls, p.BT, p.N, D);
        L.check("cls_row");
      }
      Epi e = ep(x, D, nullptr);
      e.out_f32 = 1; e.map = g.no_cls ? MAP_LINEAR : MAP_TOKENS; e.map_p = p.P;   // no cls token: token row = patch row
      e.rowbias = wf("patch.pos", (size_t)p.P * D);
      e.rb_div = 1; e.rb_mod = p.P; e.rb_ld = D;
      linear(A0, p.Mp, KPATCH, "patch.w", D, e);
    }
    snapshot("tokens0", x, true, p.M, D, D);
    // ---- encoder blocks (block.py:110-151)
    void* xn = buf("xn");
    void* qkv = buf("qkv");
    void* ao = buf("ao");
    void* hb = buf("h");
    int tap_i = 0;
    // ViT-S (D = 384) on the tensor-core path: proj / fc2 run as row-owning GEMMs whose epilogue also emits the
    // LayerNorm'ed operand of the NEXT GEMM (gemm_ln.cuh), so only the very first norm1 and the four tap norms remain
    // separate launches.  xn_ready: xn already holds norm1_i(x) (written by fc2 of block i-1).
    const bool fuse_ln = tc() && gemm_ln_supported(dt, D, D) && gemm_ln_supported(dt, D, 4 * D);
    bool xn_ready = false;
    for (int i = 0; i < g.depth && L.ok(); ++i) {
      const std::string n = "blk" + std::to_string(i) + ".";
      if (!xn_ready) layernorm(L, dt, x, wf(n + "ln1.w", D), wf(n + "ln1.b", D), xn, p.M, D, 1e-6f);
      xn_ready = false;
      linear(xn, p.M, D, n + "qkv.w", 3 * D, ep(qkv, 3 * D, wf(n + "qkv.b", 3 * D)));
      attention(L, dt, eng, qkv, ao, p.BT, p.N, g.heads);
      if (fuse_ln) {
        // x += ls1(proj(ao)); xn = norm2(x)      (LayerScale folded into proj.w / proj.b)
        L.tag = "blk.proj";
        gemm_ln(L, dt, ao, wt(n + "proj.w", (size_t)D * D), wf(n + "proj.b", D), x, xn, wf(n + "ln2.w", D), wf(n + "ln2.b", D), 1e-6f,
                (int)p.M, D, D, 1);
        L.tag.clear();
      } else {
        Epi e = ep(x, D, wf(n + "proj.b", D));  // LayerScale folded into proj.w / proj.b
        e.out_f32 = 1; e.res1 = x; e.res1_f32 = 1; e.ld_res1 = D;
        linear(ao, p.M, D, n + "proj.w", D, e);
        layernorm(L, dt, x, wf(n + "ln2.w", D), wf(n + "ln2.b", D), xn, p.M, D, 1e-6f);
      }
      {
        Epi e = ep(hb, 4 * D, wf(n + "fc1.b", 4 * D));  // LoRA merged into fc1.w (mylora/layers.py:384-393)
        e.act = ACT_GELU;
        linear(xn, p.M, D, n + "fc1.w", 4 * D, e);
      }
      if (fuse_ln) {
        // x += ls2(fc2(h)); xn = norm1 of the NEXT block, unless this block ends with a residual bottleneck (which
        // changes x again) or is the last one
        const bool next_ln = (i + 1 < g.depth) && !(g.res_blocks & (1 << i));
        const std::string nn = "blk" + std::to_string(i + 1) + ".";
        L.tag = "blk.fc2";
        gemm_ln(L, dt, hb, wt(n + "fc2.w", (size_t)D * 4 * D), wf(n + "fc2.b", D), x, xn, next_ln ? wf(nn + "ln1.w", D) : nullptr,
                next_ln ? wf(nn + "ln1.b", D) : nullptr, 1e-6f, (int)p.M, D, 4 * D, next_ln ? 1 : 0);
        L.tag.clear();
        xn_ready = next_ln;
      } else {
        Epi e = ep(x, D, wf(n + "fc2.b", D));
        e.out_f32 = 1; e.res1 = x; e.res1_f32 = 1; e.ld_res1 = D;
        linear(hb, p.M, 4 * D, n + "fc2.w", D, e);
      }
      if (g.res_blocks & (1 << i)) res_block(n, x);
      if (i == 0) snapshot("block0", x, true, p.M, D, D);
      if (tap_i < 4 && i == g.taps[tap_i]) {
        char tn[16];
        snprintf(tn, sizeof tn, "tap%d", tap_i);
        // final norm on the tap + cls split (vision_transformer.py:318-321)
        layernorm(L, dt, x, wf("norm.w", D), wf("norm.b", D), buf(tn), p.Mp, D, 1e-6f, g.no_cls ? 0 : p.N, g.no_cls ? 0 : 1);
        snapshot(tn, buf(tn), false, p.Mp, D, D);
        if (g.use_clstoken) {
          // readout projects (dpt.py:92-99; dpt_pyramid.py:54-57): tap' = GELU(Linear(2D, D)([token | class token])) =
          // GELU(token W1^T + rb[frame]) with the per-frame row bias rb = class token W2^T + b.  The class token is row 0
          // of the frame after the final norm (without a cls token: its first patch token, as in the reference).
          char cn[16], rn_[16], on[16];
          snprintf(cn, sizeof cn, "tapc%d", tap_i);
          snprintf(rn_, sizeof rn_, "rorb%d", tap_i);
          snprintf(on, sizeof on, "tapr%d", tap_i);
          const std::string ro = "ro" + std::to_string(tap_i) + ".";
          layernorm(L, dt, x, wf("norm.w", D), wf("norm.b", D), buf(cn), p.BT, D, 1e-6f, p.N, -1);
          {
            Epi e = ep(buf(rn_), D, wf(ro + "b", D));
            e.out_f32 = 1;
            linear(buf(cn), p.BT, D, ro + "w2", D, e);
          }
          {
            Epi e = ep(buf(on), D, nullptr);
            e.rowbias = (const float*)buf(rn_);
            e.rb_div = p.P; e.rb_mod = p.BT; e.rb_ld = D;
            e.act = ACT_GELU;
            linear(buf(tn), p.Mp, D, ro + "w1", D, e);
          }
        }
        ++tap_i;
      }
    }
    if (tap_i != 4) L.fail(EDV_ERR_ARG, "taps must be increasing block indices < depth");
    // ---- DPT head (dpt_pyramid.py:51-113)
    const int F_ = g.features;
    void* L1 = buf("L1");
    void* L2 = buf("L2");
    void* L3 = buf("L3");
    void* L4p = buf("L4p");
    void* L4 = buf("L4");
    // endodac (models/endodac/endodac.py:93-127) is this head without the four temporal modules
    const bool mm_on = !g.no_motion;
    void* L3m = mm_on ? buf("L3m") : L3;
    void* L4m = mm_on ? buf("L4m") : L4;
    void *l1r = buf("l1r"), *l2r = buf("l2r"), *l3r = buf("l3r"), *l4r = buf("l4r");
    void *l1rr = buf("l1rr"), *l2rr = buf("l2rr"), *l3rr = buf("l3rr"), *l4rr = buf("l4rr");
    // The decoder is a DAG: paths 1-3 (reassemble -> [temporal module 0] -> layer_rn) only meet the deep path at
    // their fusion blocks.  The deep path (path 4 -> refinenet4 -> module 2 -> refinenet3 -> module 3 -> ...) is a
    // chain of small, latency-bound launches on 19 x 19 / 37 x 37 maps that leaves most SMs idle, so paths 1-3 run
    // beside it on the side stream (same kernels, same buffers per tensor: bit-identical to the serial order).
    fork_side();
    {
      // projects[0] (1x1) merged with resize_layers[0] (ConvT k4 s4): one GEMM + pixel shuffle
      Epi e = ep(L1, p.Cp[0], wf("proj0.b", 16 * p.Cp[0]));
      e.map = MAP_PIXSHUF; e.ps_k = 4; e.ps_h = p.ph; e.ps_w = p.pw; e.ps_c = p.Cp[0];
      linear(buf(g.use_clstoken ? "tapr0" : "tap0"), p.Mp, D, "proj0.w", 16 * p.Cp[0], e);
    }
    {
      Epi e = ep(L2, p.Cp[1], wf("proj1.b", 4 * p.Cp[1]));
      e.map = MAP_PIXSHUF; e.ps_k = 2; e.ps_h = p.ph; e.ps_w = p.pw; e.ps_c = p.Cp[1];
      linear(buf(g.use_clstoken ? "tapr1" : "tap1"), p.Mp, D, "proj1.w", 4 * p.Cp[1], e);
    }
    linear(buf(g.use_clstoken ? "tapr2" : "tap2"), p.Mp, D, "proj2.w", p.Cp[2], ep(L3, p.Cp[2], wf("proj2.b", p.Cp[2])));
    if (mm_on) motion(0, L3, L3m, par ? "mmb." : "mm.");
    // scratch.layer{1-4}_rn (3x3, no bias) -> F channels, plus relu copies for the RCUs
    {
      Epi e = ep(l3r, F_, nullptr); e.out_relu = l3rr;
      conv3(L3m, p.BT, p.ph, p.pw, p.Cp[2], "rn3.w", F_, e);
      e = ep(l2r, F_, nullptr); e.out_relu = l2rr;
      conv3(L2, p.BT, 2 * p.ph, 2 * p.pw, p.Cp[1], "rn2.w", F_, e);
      e = ep(l1r, F_, nullptr); e.out_relu = l1rr;
      conv3(L1, p.BT, 4 * p.ph, 4 * p.pw, p.Cp[0], "rn1.w", F_, e);
    }
    back_to_main();
    linear(buf(g.use_clstoken ? "tapr3" : "tap3"), p.Mp, D, "proj3.w", p.Cp[3], ep(L4p, p.Cp[3], wf("proj3.b", p.Cp[3])));
    {
      // resize_layers[3]: 3x3 stride 2 pad 1 (dpt.py:85-90) = explicit im2col + GEMM
      const long long Mo = (long long)p.BT * p.ph2 * p.pw2;
      if (tc()) {
        void* col = buf("col");
        if (L.ok()) {
          long long tot = Mo * 9 * (p.Cp[3] / 8);
          EDV_DISPATCH_T(dt, { edv::launch_k(im2col3x3_kernel<T>, dim3(nblk(tot, 256)), dim3(256), 0, L.stream, (const T*)L4p, (T*)col, p.BT, p.ph, p.pw, p.Cp[3], p.ph2, p.pw2, 2); });
          L.check("im2col");
        }
        linear(col, Mo, 9 * p.Cp[3], "resize3.w", p.Cp[3], ep(L4, p.Cp[3], wf("resize3.b", p.Cp[3])));
      } else {
        GemmArgs a;
        a.A = L4p; a.W = wt("resize3.w", (size_t)p.Cp[3] * 9 * p.Cp[3]); a.M = (int)Mo; a.N = p.Cp[3]; a.K = 9 * p.Cp[3];
        a.e = ep(L4, p.Cp[3], wf("resize3.b", p.Cp[3]));
        a.conv = true; a.F = p.BT; a.H = p.ph; a.Wd = p.pw; a.C = p.Cp[3]; a.stride = 2;
        if (L.ok()) gemm(L, dt, eng, a);
      }
    }
    if (mm_on) motion(1, L4, L4m);
    {
      Epi e = ep(l4r, F_, nullptr); e.out_relu = l4rr;
      conv3(L4m, p.BT, p.ph2, p.pw2, p.Cp[3], "rn4.w", F_, e);
    }
    snapshot("layer1", L1, false, (long long)p.BT * 16 * p.P, p.Cp[0], g.out_channels[0]);
    snapshot("layer2", L2, false, (long long)p.BT * 4 * p.P, p.Cp[1], g.out_channels[1]);
    snapshot("layer3", L3, false, p.Mp, p.Cp[2], g.out_channels[2]);
    snapshot("layer4", L4, false, (long long)p.BT * p.ph2 * p.pw2, p.Cp[3], g.out_channels[3]);
    snapshot("mm0", L3m, false, p.Mp, p.Cp[2], g.out_channels[2]);
    snapshot("mm1", L4m, false, (long long)p.BT * p.ph2 * p.pw2, p.Cp[3], g.out_channels[3]);
    void *p4 = buf("p4"), *p3 = buf("p3"), *p2 = buf("p2"), *p1 = buf("p1");
    void *p4m = mm_on ? buf("p4m") : p4, *p3m = mm_on ? buf("p3m") : p3;
    fusion(4, l4r, l4rr, nullptr, nullptr, p.ph2, p.pw2, p.ph, p.pw, p4);
    snapshot("path4_pre", p4, false, p.Mp, F_, F_);
    if (mm_on) motion(2, p4, p4m);
    join_side();   // refinenet3 is the first consumer of the side stream's layer{1,2,3}_rn maps
    fusion(3, p4m, nullptr, l3r, l3rr, p.ph, p.pw, 2 * p.ph, 2 * p.pw, p3);
    if (mm_on) motion(3, p3, p3m);
    snapshot("path3", p3m, false, (long long)p.BT * 4 * p.P, F_, F_);
    fusion(2, p3m, nullptr, l2r, l2rr, 2 * p.ph, 2 * p.pw, 4 * p.ph, 4 * p.pw, p2);
    fusion(1, p2, nullptr, l1r, l1rr, 4 * p.ph, 4 * p.pw, 8 * p.ph, 8 * p.pw, p1);
    snapshot("path1", p1, false, (long long)p.BT * 64 * p.P, F_, F_);
    // ---- disparity outputs
    float* d[4];
    for (int s = 0; s < 4; ++s) d[s] = disp[s] ? disp[s] : (float*)buf(s == 0 ? "disp0" : s == 1 ? "disp1" : s == 2 ? "disp2" : "disp3");
    if (!g.conv_head) {
      disp_head("oc1", "oc2a", "oc2b", p1, 8 * p.ph, 8 * p.pw, p.out_h[0], p.out_w[0], 0.f, d[0]);
      for (int s = 1; s < 4; ++s) resize_f32(L, d[s - 1], d[s], p.BT, p.out_h[s - 1], p.out_w[s - 1], p.out_h[s], p.out_w[s]);
      if (g.out_sigmoid && L.ok()) {
        for (int s = 0; s < 4; ++s) {
          long long n = (long long)p.BT * p.out_h[s] * p.out_w[s];
          sigmoid_inplace_kernel<<<nblk(n, 256), 256, 0, L.stream>>>(d[s], n);
          L.check("sigmoid");
        }
      }
    } else {
      const float sg = g.inv_sigmoid ? -1.f : 1.f;
      disp_head("cd4.c0", "cd4.c2", "cd4.c4", p4m, p.ph, p.pw, p.out_h[3], p.out_w[3], sg, d[3]);
      disp_head("cd3.c0", "cd3.c2", "cd3.c4", p3m, 2 * p.ph, 2 * p.pw, p.out_h[2], p.out_w[2], sg, d[2]);
      disp_head("cd2.c0", "cd2.c2", "cd2.c4", p2, 4 * p.ph, 4 * p.pw, p.out_h[1], p.out_w[1], sg, d[1]);
      disp_head("cd1.c0", "cd1.c2", "cd1.c4", p1, 8 * p.ph, 8 * p.pw, p.out_h[0], p.out_w[0], sg, d[0]);
    }
    if (resized) resize_f32(L, d[0], resized, p.BT, p.out_h[0], p.out_w[0], out_h, out_w);
    c->last_launches = L.count;
    if (!L.ok()) c->err = L.err;
    return L.status;
  }

  // ResBottleneckBlock on the patch tokens (block.py:146-150; layers/utils.py:143-152)
  void res_block(const std::string& n, float* x) {
    const Plan& p = c->plan;
    const int D = c->cfg.dim, bc = D / 8, bcp = round_up(bc, 64);
    void* pt = buf("rb.pt");
    void* t1 = buf("rb.t1");
    void* t2 = buf("rb.t2");
    void* t3 = buf("rb.t3");
    if (!L.ok()) return;
    EDV_DISPATCH_T(dt, {
      tokens_to_patches_kernel<T><<<nblk(p.Mp * (D / 4), 256), 256, 0, L.stream>>>(x, (T*)pt, p.Mp, p.P, D, c->cfg.no_cls ? 0 : 1);
    });
    L.check("tokens_to_patches");
    linear(pt, p.Mp, D, n + "res.c1.w", bcp, ep(t1, bcp, nullptr));
    if (L.ok()) {
      EDV_DISPATCH_T(dt, { rowln_act_kernel<T><<<nblk(p.Mp * 32, 256), 256, 0, L.stream>>>((const T*)t1, wf(n + "res.n1.w", bcp), wf(n + "res.n1.b", bcp), (T*)t2, p.Mp, bcp, bc, 1e-6f, 1); });
      L.check("res ln1");
    }
    conv3(t2, p.BT, p.ph, p.pw, bcp, n + "res.c2.w", bcp, ep(t1, bcp, nullptr));
    if (L.ok()) {
      EDV_DISPATCH_T(dt, { rowln_act_kernel<T><<<nblk(p.Mp * 32, 256), 256, 0, L.stream>>>((const T*)t1, wf(n + "res.n2.w", bcp), wf(n + "res.n2.b", bcp), (T*)t2, p.Mp, bcp, bc, 1e-6f, 1); });
      L.check("res ln2");
    }
    linear(t2, p.Mp, bcp, n + "res.c3.w", D, ep(t3, D, nullptr));
    if (L.ok()) {
      EDV_DISPATCH_T(dt, { resblock_add_kernel<T><<<nblk(p.Mp * 32, 256), 256, 0, L.stream>>>(x, (const T*)t3, wf(n + "res.n3.w", D), wf(n + "res.n3.b", D), p.Mp, p.P, D, 1e-6f, c->cfg.no_cls ? 0 : 1); });
      L.check("res add");
    }
  }
};

int set_err(edv_ctx* c, int code, const char* fmt, ...) {
  char b[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(b, sizeof b, fmt, ap);
  va_end(ap);
  if (c) c->err = b;
  else g_create_error = b;
  return code;
}

}  // namespace

// =========================================================================================
// C ABI
// =========================================================================================
extern "C" {

int edv_abi_version(void) { return EDV_ABI_VERSION; }

int edv_create(const edv_config* cfg, edv_ctx** out) {
  if (!cfg || !out) return set_err(nullptr, EDV_ERR_ARG, "edv_create: null argument");
  *out = nullptr;
  if (cfg->dim <= 0 || cfg->dim % 64 != 0 || cfg->heads <= 0 || cfg->dim != cfg->heads * 64)
    return set_err(nullptr, EDV_ERR_ARG, "edv_create: dim must equal heads*64 (got dim=%d heads=%d)", cfg->dim, cfg->heads);
  if (cfg->dim > 1024) return set_err(nullptr, EDV_ERR_ARG, "edv_create: dim > 1024 unsupported");
  if (cfg->depth <= 0 || cfg->depth > 31) return set_err(nullptr, EDV_ERR_ARG, "edv_create: bad depth %d", cfg->depth);
  if (cfg->features % 64 != 0 || cfg->features <= 0)
    return set_err(nullptr, EDV_ERR_ARG, "edv_create: features must be a multiple of 64");
  if (cfg->out_channels[2] % 64 != 0 || cfg->out_channels[3] % 64 != 0)
    return set_err(nullptr, EDV_ERR_ARG, "edv_create: out_channels[2:4] must be multiples of 64 (GroupNorm(32) inputs)");
  if (cfg->num_frames < 1 || cfg->num_frames > 32)
    return set_err(nullptr, EDV_ERR_ARG, "edv_create: num_frames must be in [1,32]");
  if (cfg->dtype < EDV_F32 || cfg->dtype > EDV_F16) return set_err(nullptr, EDV_ERR_ARG, "edv_create: bad dtype");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return set_err(nullptr, EDV_ERR_NO_DEVICE, "edv_create: no CUDA device (this library has no CPU fallback)");
  }
  int dev = 0;
  cudaGetDevice(&dev);
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, dev);
  if (prop.major != 10)
    return set_err(nullptr, EDV_ERR_NO_DEVICE, "edv_create: device is sm_%d%d, kernels are built for sm_100a only", prop.major, prop.minor);
  edv_ctx* c = new edv_ctx();
  c->cfg = *cfg;
  if (const char* env = getenv("EDV_GRAPH")) c->graph_mode = atoi(env) != 0;
  if (const char* env = getenv("EDV_BRANCH")) c->branch_mode = atoi(env) != 0;
  *out = c;
  return EDV_OK;
}

void edv_destroy(edv_ctx* ctx) { delete ctx; }

const char* edv_last_error(const edv_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int edv_set_weight(edv_ctx* ctx, const char* name, const void* dev_ptr, size_t bytes) {
  if (!ctx || !name || !dev_ptr) return set_err(ctx, EDV_ERR_ARG, "edv_set_weight: null argument");
  if (((uintptr_t)dev_ptr & 15) != 0) return set_err(ctx, EDV_ERR_ARG, "edv_set_weight: '%s' must be 16-byte aligned", name);
  auto it = ctx->weights.find(name);
  if (it == ctx->weights.end() || it->second.ptr != dev_ptr || it->second.bytes != bytes) ctx->drop_graphs();   // pointers are baked into captured graphs
  ctx->weights[name] = WeightRef{dev_ptr, bytes};
  return EDV_OK;
}

int edv_set_debug(edv_ctx* ctx, int on) {
  if (!ctx) return EDV_ERR_ARG;
  ctx->debug = on;
  ctx->plan.valid = false;
  ctx->drop_graphs();
  return EDV_OK;
}

int edv_plan(edv_ctx* ctx, int B, int T, int H, int W, int net_h, int net_w, size_t* workspace_bytes) {
  if (!ctx || !workspace_bytes) return set_err(ctx, EDV_ERR_ARG, "edv_plan: null argument");
  const edv_config& g = ctx->cfg;
  if (B < 1 || T < 1 || T > g.num_frames)
    return set_err(ctx, EDV_ERR_ARG, "edv_plan: T=%d must be in [1,num_frames=%d] (PE table, motion_module.py:185-197)", T, g.num_frames);
  if (net_h % 14 != 0 || net_w % 14 != 0 || net_h < 14 || net_w < 14)
    return set_err(ctx, EDV_ERR_ARG, "edv_plan: network resolution %dx%d must be multiples of 14 (patch_embed.py:72-73)", net_h, net_w);
  if (H < 1 || W < 1) return set_err(ctx, EDV_ERR_ARG, "edv_plan: bad frame size");
  Plan p;
  p.B = B; p.T = T; p.H = H; p.W = W; p.h = net_h; p.w = net_w;
  p.BT = B * T; p.ph = net_h / 14; p.pw = net_w / 14; p.P = p.ph * p.pw; p.N = p.P + (g.no_cls ? 0 : 1);
  p.M = (long long)p.BT * p.N; p.Mp = (long long)p.BT * p.P;
  p.ph2 = (p.ph - 1) / 2 + 1; p.pw2 = (p.pw - 1) / 2 + 1;
  if (p.M * 4LL * g.dim > 2000000000LL * 4) return set_err(ctx, EDV_ERR_ARG, "edv_plan: clip batch too large for 32-bit row indexing");
  for (int i = 0; i < 4; ++i) p.Cp[i] = round_up(g.out_channels[i], 64);
  if (g.res_blocks) {
    if (g.dim % 8 != 0) return set_err(ctx, EDV_ERR_ARG, "edv_plan: residual blocks need dim %% 8 == 0");
  }
  const int F_ = g.features, Fh = F_ / 2;
  p.mm[0] = MMPlan{p.Cp[2], p.ph, p.pw};
  p.mm[1] = MMPlan{p.Cp[3], p.ph2, p.pw2};
  p.mm[2] = MMPlan{F_, p.ph, p.pw};
  p.mm[3] = MMPlan{F_, 2 * p.ph, 2 * p.pw};
  for (int j = 0; j < 4 && !g.no_motion; ++j) {
    int hd = p.mm[j].C / 8;
    if (!(hd == 8 || hd == 24 || hd == 32 || hd == 48 || hd == 128))
      return set_err(ctx, EDV_ERR_ARG, "edv_plan: temporal head dim %d unsupported (8,24,32,48,128)", hd);
  }
  if (!g.conv_head) {
    p.out_h[0] = net_h; p.out_w[0] = net_w;
    for (int s = 1; s < 4; ++s) { p.out_h[s] = p.out_h[s - 1] / 2; p.out_w[s] = p.out_w[s - 1] / 2; }  // scale_factor=0.5 -> floor
  } else {
    p.out_h[0] = 16 * p.ph; p.out_w[0] = 16 * p.pw;   // HeadDepth upsamples x2 (layers.py:211)
    p.out_h[1] = 8 * p.ph; p.out_w[1] = 8 * p.pw;
    p.out_h[2] = 4 * p.ph; p.out_w[2] = 4 * p.pw;
    p.out_h[3] = 2 * p.ph; p.out_w[3] = 2 * p.pw;
  }
  for (int s = 0; s < 4; ++s)
    if (p.out_h[s] < 1 || p.out_w[s] < 1) return set_err(ctx, EDV_ERR_ARG, "edv_plan: resolution too small for the 4-level pyramid");

  const size_t es = dtype_size(g.dtype);
  size_t off = 0;
  auto add = [&](const char* name, size_t bytes, int elem = 0) {
    Buf b;
    b.off = off;
    b.bytes = bytes;
    b.elem = elem ? elem : (int)es;
    p.bufs[name] = b;
    off += (bytes + 1023) & ~(size_t)1023;
  };
  const int D = g.dim;
  const bool simt = (g.dtype == EDV_F32) || g.engine == EDV_ENGINE_SIMT;
  add("A0", (size_t)p.Mp * KPATCH * es);
  add("x", (size_t)p.M * D * 4, 4);
  add("xn", (size_t)p.M * D * es);
  add("qkv", (size_t)p.M * 3 * D * es);
  add("ao", (size_t)p.M * D * es);
  add("h", (size_t)p.M * 4 * D * es);
  for (int i = 0; i < 4; ++i) {
    char n[8];
    snprintf(n, sizeof n, "tap%d", i);
    add(n, (size_t)p.Mp * D * es);
    if (g.use_clstoken) {
      char m[16];
      snprintf(m, sizeof m, "tapc%d", i);
      add(m, (size_t)p.BT * D * es);
      snprintf(m, sizeof m, "rorb%d", i);
      add(m, (size_t)p.BT * D * 4, 4);
      snprintf(m, sizeof m, "tapr%d", i);
      add(m, (size_t)p.Mp * D * es);
    }
  }
  if (g.res_blocks) {
    const int bcp = round_up(D / 8, 64);
    add("rb.pt", (size_t)p.Mp * D * es);
    add("rb.t1", (size_t)p.Mp * bcp * es);
    add("rb.t2", (size_t)p.Mp * bcp * es);
    add("rb.t3", (size_t)p.Mp * D * es);
  }
  const size_t px1 = (size_t)p.BT * 16 * p.P, px2 = (size_t)p.BT * 4 * p.P, px3 = (size_t)p.Mp, px4 = (size_t)p.BT * p.ph2 * p.pw2;
  const size_t px0 = (size_t)p.BT * 64 * p.P;  // 8ph x 8pw
  add("L1", px1 * p.Cp[0] * es);
  add("L2", px2 * p.Cp[1] * es);
  add("L3", px3 * p.Cp[2] * es);
  add("L4p", px3 * p.Cp[3] * es);
  add("L4", px4 * p.Cp[3] * es);
  if (!simt) add("col", px4 * 9 * p.Cp[3] * es);
  if (!g.no_motion) {
    add("L3m", px3 * p.Cp[2] * es);
    add("L4m", px4 * p.Cp[3] * es);
  }
  // motion-module scratch, sized for the largest of the four modules
  size_t mmC = 0, mm3 = 0, mm4 = 0, mm8 = 0;
  for (int j = 0; j < 4; ++j) {
    size_t rows = (size_t)p.BT * p.mm[j].h * p.mm[j].w, C = p.mm[j].C;
    mmC = std::max(mmC, rows * C);
    mm3 = std::max(mm3, rows * 3 * C);
    mm4 = std::max(mm4, rows * 4 * C);
    mm8 = std::max(mm8, rows * 8 * C);
  }
  if (!g.no_motion) {
    add("mm.stats", (size_t)p.BT * 32 * (1 + GN_MAX_SPLIT) * sizeof(float2), 8);
    add("mm.gn", mmC * es);
    add("mm.hs", mmC * 4, 4);
    add("mm.ln", mmC * es);
    add("mm.qkv", mm3 * es);
    add("mm.att", mmC * es);
    add("mm.gg", mm4 * es);
    add("mm.hsT", mmC * es);
    // second scratch family for module 0, which runs on the side stream while module 1 runs on the main one
    const size_t r0 = (size_t)p.BT * p.mm[0].h * p.mm[0].w * p.mm[0].C;
    add("mmb.stats", (size_t)p.BT * 32 * (1 + GN_MAX_SPLIT) * sizeof(float2), 8);
    add("mmb.gn", r0 * es);
    add("mmb.hs", r0 * 4, 4);
    add("mmb.ln", r0 * es);
    add("mmb.qkv", 3 * r0 * es);
    add("mmb.att", r0 * es);
    add("mmb.gg", 4 * r0 * es);
    add("mmb.hsT", r0 * es);
  }
  if (simt && !g.no_motion) {
    add("mm.gg2", mm8 * es);
    add("mmb.gg2", 8 * (size_t)p.BT * p.mm[0].h * p.mm[0].w * p.mm[0].C * es);
  }
  add("l1r", px1 * F_ * es); add("l1rr", px1 * F_ * es);
  add("l2r", px2 * F_ * es); add("l2rr", px2 * F_ * es);
  add("l3r", px3 * F_ * es); add("l3rr", px3 * F_ * es);
  add("l4r", px4 * F_ * es); add("l4rr", px4 * F_ * es);
  // refinenet scratch at the largest input resolution (refinenet1 runs at 4ph x 4pw)
  add("ref.tmp", px1 * F_ * es);
  add("ref.s", px1 * F_ * es);
  add("ref.sr", px1 * F_ * es);
  add("ref.u", px1 * F_ * es);
  add("ref.v", px1 * F_ * es);
  add("p4", px3 * F_ * es); add("p4m", px3 * F_ * es);
  add("p3", px2 * F_ * es); add("p3m", px2 * F_ * es);
  add("p2", px1 * F_ * es);
  add("p1", px0 * F_ * es);
  // disparity head scratch: conv at up to 8ph x 8pw, upsample target up to out_h[0] x out_w[0]
  const size_t pxo = (size_t)p.BT * p.out_h[0] * p.out_w[0];
  add("head.o1", px0 * Fh * es);
  const bool fused_head = !simt && head_fused_supported(g.dtype, Fh);   // the upsampled map never exists in HBM then
  if (!fused_head) add("head.up", pxo * Fh * es);
  if (simt) add("head.t32", pxo * 32 * es);
  for (int s = 0; s < 4; ++s) {
    char n[8];
    snprintf(n, sizeof n, "disp%d", s);
    add(n, (size_t)p.BT * p.out_h[s] * p.out_w[s] * 4, 4);
  }
  if (ctx->debug) {
    auto tap = [&](const char* name, long long rows, int cols) {
      DebugTap t;
      t.rows = rows;
      t.cols = cols;
      t.buf.off = off;
      t.buf.bytes = (size_t)rows * cols * 4;
      off += (t.buf.bytes + 1023) & ~(size_t)1023;
      p.taps[name] = t;
    };
    tap("tokens0", p.M, D);
    tap("block0", p.M, D);
    for (int i = 0; i < 4; ++i) {
      char n[8];
      snprintf(n, sizeof n, "tap%d", i);
      tap(n, p.Mp, D);
    }
    tap("layer1", px1, g.out_channels[0]);
    tap("layer2", px2, g.out_channels[1]);
    tap("layer3", px3, g.out_channels[2]);
    tap("layer4", px4, g.out_channels[3]);
    tap("mm0", px3, g.out_channels[2]);
    tap("mm1", px4, g.out_channels[3]);
    tap("path4_pre", px3, F_);
    tap("path3", px2, F_);
    tap("path1", px0, F_);
  }
  p.total = off + 1024;
  p.valid = true;
  ctx->drop_graphs();
  ctx->plan = p;
  *workspace_bytes = p.total;
  return EDV_OK;
}

// the captured forward leaves the disparity pyramid in the plan's buffers: hand it to the caller's tensors with ONE
// launch for all four levels (four cudaMemcpyAsync cost ~15 us of launch gaps at the reference's resolution)
struct PyramidCopy {
  const float4* src[4];
  float4* dst[4];
  unsigned long long n4[4];    // float4 elements per level (every level is a multiple of 4 floats: checked below)
  unsigned long long start[5]; // prefix sums of n4
};
__global__ void __launch_bounds__(256) copy_pyramid_kernel(PyramidCopy c) {
  pdl_launch();
  pdl_wait();
  const unsigned long long total = c.start[4];
  for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (unsigned long long)gridDim.x * blockDim.x) {
    const int s = i >= c.start[3] ? 3 : i >= c.start[2] ? 2 : i >= c.start[1] ? 1 : 0;
    const unsigned long long k = i - c.start[s];
    c.dst[s][k] = c.src[s][k];
  }
}
static int copy_pyramid_out(edv_ctx* ctx, float* const disp[4], void* workspace_dev, cudaStream_t st) {
  static const char* names[4] = {"disp0", "disp1", "disp2", "disp3"};
  PyramidCopy c;
  c.start[0] = 0;
  bool vec = true, any = false;
  size_t bytes[4];
  const unsigned char* src[4];
  for (int s = 0; s < 4; ++s) {
    c.src[s] = nullptr; c.dst[s] = nullptr; c.n4[s] = 0; bytes[s] = 0; src[s] = nullptr;
    if (disp[s]) {
      auto it = ctx->plan.bufs.find(names[s]);
      if (it == ctx->plan.bufs.end()) return set_err(ctx, EDV_ERR_STATE, "edv_forward: internal disparity buffer missing");
      const size_t n = (size_t)ctx->plan.BT * ctx->plan.out_h[s] * ctx->plan.out_w[s];
      bytes[s] = n * sizeof(float);
      src[s] = (const unsigned char*)workspace_dev + it->second.off;
      if ((n & 3) || ((uintptr_t)disp[s] & 15) || ((uintptr_t)src[s] & 15)) vec = false;
      c.src[s] = (const float4*)src[s]; c.dst[s] = (float4*)disp[s]; c.n4[s] = n / 4;
      any = true;
    }
    c.start[s + 1] = c.start[s] + c.n4[s];
  }
  if (!any) return EDV_OK;
  if (vec) {
    const unsigned long long total = c.start[4];
    const unsigned blocks = (unsigned)std::min<unsigned long long>((total + 255) / 256, 8ull * num_sms());
    copy_pyramid_kernel<<<blocks, 256, 0, st>>>(c);   // plain launch: fully ordered behind the graph
    if (cudaGetLastError() != cudaSuccess) return set_err(ctx, EDV_ERR_CUDA, "edv_forward: copy of the disparity pyramid failed");
    return EDV_OK;
  }
  for (int s = 0; s < 4; ++s)   // odd sizes / unaligned caller tensors: plain copies
    if (disp[s] && cudaMemcpyAsync(disp[s], src[s], bytes[s], cudaMemcpyDeviceToDevice, st) != cudaSuccess)
      return set_err(ctx, EDV_ERR_CUDA, "edv_forward: copy of the disparity pyramid failed: %s", cudaGetErrorString(cudaGetLastError()));
  return EDV_OK;
}

static int forward_common(edv_ctx* ctx, const void* frames, bool u8, float* const disp_dev[4], float* resized_dev,
                          int out_h, int out_w, void* workspace_dev, void* stream) {
  if (!ctx || !frames || !workspace_dev) return set_err(ctx, EDV_ERR_ARG, "edv_forward: null argument");
  if (!ctx->plan.valid) return set_err(ctx, EDV_ERR_STATE, "edv_forward: call edv_plan first");
  if (((uintptr_t)workspace_dev & 1023) != 0) return set_err(ctx, EDV_ERR_ARG, "edv_forward: workspace must be 1024-byte aligned");
  if (resized_dev && (out_h < 1 || out_w < 1)) return set_err(ctx, EDV_ERR_ARG, "edv_forward: bad resize target");
  if (u8 && (ctx->plan.H != ctx->plan.h || ctx->plan.W != ctx->plan.w))
    return set_err(ctx, EDV_ERR_ARG, "edv_forward_u8: frames must already be at network resolution");
  float* none[4] = {nullptr, nullptr, nullptr, nullptr};
  float* const* disp = disp_dev ? disp_dev : none;
  cudaStream_t st = (cudaStream_t)stream;
  const bool graphable = ctx->graph_mode && !ctx->prof.on && !ctx->debug && ctx->plan_warm;
  if (!graphable) {
    Fwd f(ctx, workspace_dev, st);
    const int rc = f.run(frames, u8, disp, resized_dev, out_h, out_w);
    if (rc == EDV_OK) ctx->plan_warm = true;
    return rc;
  }
  GraphEntry key;
  key.frames = frames; key.resized = resized_dev; key.workspace = workspace_dev;
  key.u8 = u8; key.out_h = resized_dev ? out_h : 0; key.out_w = resized_dev ? out_w : 0;
  ++ctx->graph_clock;
  for (GraphEntry& g : ctx->graphs) {
    if (!g.same(key)) continue;
    g.last_use = ctx->graph_clock;
    ctx->last_launches = g.launches;
    if (cudaGraphLaunch(g.exec, st) != cudaSuccess) return set_err(ctx, EDV_ERR_CUDA, "edv_forward: cudaGraphLaunch failed: %s", cudaGetErrorString(cudaGetLastError()));
    return copy_pyramid_out(ctx, disp, workspace_dev, st);
  }
  // A capture costs about as much as a forward at the reference's resolution, so a pointer set is captured only the
  // SECOND time it comes by: a caller whose buffers never repeat (fresh tensors from a cold or fragmented allocator,
  // outputs pinned by record_stream) runs eagerly and pays nothing, a steady caller replays from its third call on.
  {
    bool met = false;
    for (GraphEntry& g : ctx->seen)
      if (g.same(key)) {
        met = true;
        g = ctx->seen.back();
        ctx->seen.pop_back();
        break;
      }
    if (!met) {
      key.last_use = ctx->graph_clock;
      if (ctx->seen.size() >= 4 * (size_t)edv_ctx::GRAPH_SLOTS) ctx->seen.erase(ctx->seen.begin());
      ctx->seen.push_back(key);
      Fwd f(ctx, workspace_dev, st);
      return f.run(frames, u8, disp, resized_dev, out_h, out_w);
    }
  }
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(st, &cs) != cudaSuccess || cs != cudaStreamCaptureStatusNone) {
    // the caller is capturing this stream itself: just record our launches into its graph
    cudaGetLastError();
    Fwd f(ctx, workspace_dev, st);
    return f.run(frames, u8, disp, resized_dev, out_h, out_w);
  }
  // Capture on a private stream and replay on the caller's: the capture itself executes nothing, and the caller's
  // stream is usually torch's current stream = the legacy default stream, which cudaStreamBeginCapture refuses.
  int prio_lo = 0, prio_hi = 0;
  cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);   // the captured main chain outranks the side-stream branches
  if (!ctx->cap_stream && cudaStreamCreateWithPriority(&ctx->cap_stream, cudaStreamNonBlocking, prio_hi) != cudaSuccess) {
    ctx->graph_note = std::string("cudaStreamCreateWithPriority: ") + cudaGetErrorString(cudaGetLastError());
    ctx->cap_stream = nullptr;
    ctx->graph_mode = 0;
    Fwd f(ctx, workspace_dev, st);
    return f.run(frames, u8, disp, resized_dev, out_h, out_w);
  }
  cudaStream_t cap = ctx->cap_stream;
  cudaError_t be = cudaStreamBeginCapture(cap, cudaStreamCaptureModeThreadLocal);
  if (be != cudaSuccess) {
    ctx->graph_note = std::string("cudaStreamBeginCapture: ") + cudaGetErrorString(be);
    cudaGetLastError();
    Fwd f(ctx, workspace_dev, st);
    return f.run(frames, u8, disp, resized_dev, out_h, out_w);
  }
  int rc;
  int launches = 0;
  {
    Fwd f(ctx, workspace_dev, cap);
    rc = f.run(frames, u8, none, resized_dev, out_h, out_w);   // pyramid into the plan's own buffers (see GraphEntry)
    launches = f.L.count;
  }
  cudaGraph_t graph = nullptr;
  const cudaError_t ce = cudaStreamEndCapture(cap, &graph);
  if (rc != EDV_OK || ce != cudaSuccess || !graph) {
    if (graph) cudaGraphDestroy(graph);
    ctx->graph_note = rc != EDV_OK ? std::string("forward failed under capture: ") + ctx->err : std::string("cudaStreamEndCapture: ") + cudaGetErrorString(ce);
    cudaGetLastError();
    ctx->graph_mode = 0;   // capture is not possible in this process: stay eager (and say why in edv_graph_status)
    Fwd f(ctx, workspace_dev, st);
    return f.run(frames, u8, disp, resized_dev, out_h, out_w);
  }
  cudaGraphExec_t exec = nullptr;
  const cudaError_t ie = cudaGraphInstantiate(&exec, graph, 0);
  cudaGraphDestroy(graph);
  if (ie != cudaSuccess || !exec) {
    ctx->graph_note = std::string("cudaGraphInstantiate: ") + cudaGetErrorString(ie);
    cudaGetLastError();
    ctx->graph_mode = 0;
    Fwd f(ctx, workspace_dev, st);
    return f.run(frames, u8, disp, resized_dev, out_h, out_w);
  }
  ctx->graph_note = "ok";
  key.exec = exec;
  key.launches = launches;
  key.last_use = ctx->graph_clock;
  if ((int)ctx->graphs.size() >= edv_ctx::GRAPH_SLOTS) {
    size_t lru = 0;
    for (size_t i = 1; i < ctx->graphs.size(); ++i)
      if (ctx->graphs[i].last_use < ctx->graphs[lru].last_use) lru = i;
    cudaGraphExecDestroy(ctx->graphs[lru].exec);
    ctx->graphs[lru] = key;
  } else {
    ctx->graphs.push_back(key);
  }
  ctx->last_launches = launches;
  if (cudaGraphLaunch(exec, st) != cudaSuccess) return set_err(ctx, EDV_ERR_CUDA, "edv_forward: cudaGraphLaunch failed: %s", cudaGetErrorString(cudaGetLastError()));
  return copy_pyramid_out(ctx, disp, workspace_dev, st);
}

// 1: replay captured CUDA graphs of the planned forward (default), 0: launch every kernel from the host.
int edv_set_graph_mode(edv_ctx* ctx, int on) {
  if (!ctx) return EDV_ERR_ARG;
  ctx->graph_mode = on ? 1 : 0;
  if (!on) ctx->drop_graphs();
  return EDV_OK;
}

// number of captured graphs currently cached for this plan (tests / bench evidence)
int edv_graph_count(const edv_ctx* ctx) { return ctx ? (int)ctx->graphs.size() : 0; }

// "ok" after a successful capture, else the reason the last attempt fell back to eager launches
const char* edv_graph_status(const edv_ctx* ctx) { return ctx ? ctx->graph_note.c_str() : "null context"; }

int edv_forward(edv_ctx* ctx, const float* frames_dev, float* const disp_dev[4], float* resized_dev, int out_h,
                int out_w, void* workspace_dev, void* stream) {
  return forward_common(ctx, frames_dev, false, disp_dev, resized_dev, out_h, out_w, workspace_dev, stream);
}

int edv_forward_u8(edv_ctx* ctx, const uint8_t* frames_dev, float* const disp_dev[4], float* resized_dev, int out_h,
                   int out_w, void* workspace_dev, void* stream) {
  return forward_common(ctx, frames_dev, true, disp_dev, resized_dev, out_h, out_w, workspace_dev, stream);
}

int edv_output_shape(const edv_ctx* ctx, int scale, int* h, int* w) {
  if (!ctx || !ctx->plan.valid || scale < 0 || scale > 3 || !h || !w) return EDV_ERR_ARG;
  *h = ctx->plan.out_h[scale];
  *w = ctx->plan.out_w[scale];
  return EDV_OK;
}

int edv_launch_count(const edv_ctx* ctx) { return ctx ? ctx->last_launches : 0; }

// workspace offset of a debug tap (the Python host slices its own workspace tensor)
int edv_debug_tap(edv_ctx* ctx, const char* name, size_t* offset_bytes, long long* rows, int* cols) {
  if (!ctx || !name || !offset_bytes || !rows || !cols) return EDV_ERR_ARG;
  if (!ctx->debug || !ctx->plan.valid) return set_err(ctx, EDV_ERR_STATE, "edv_debug_tap: enable edv_set_debug before edv_plan");
  auto it = ctx->plan.taps.find(name);
  if (it == ctx->plan.taps.end()) return set_err(ctx, EDV_ERR_ARG, "edv_debug_tap: unknown tap '%s'", name);
  *offset_bytes = it->second.buf.off;
  *rows = it->second.rows;
  *cols = it->second.cols;
  return EDV_OK;
}

// Enumerate the named workspace buffers of the current plan (range / saturation checks of the 16-bit
// intermediates: the Python host views its own workspace tensor at `offset_bytes`).  Returns EDV_ERR_ARG
// past the last buffer.
int edv_plan_buffer(edv_ctx* ctx, int index, char* name, int name_cap, size_t* offset_bytes, size_t* bytes, int* elem_bytes) {
  if (!ctx || !ctx->plan.valid || index < 0 || !name || name_cap < 1 || !offset_bytes || !bytes || !elem_bytes) return EDV_ERR_ARG;
  if (index >= (int)ctx->plan.bufs.size()) return EDV_ERR_ARG;
  auto it = ctx->plan.bufs.begin();
  std::advance(it, index);
  snprintf(name, name_cap, "%s", it->first.c_str());
  *offset_bytes = it->second.off;
  *bytes = it->second.bytes;
  *elem_bytes = it->second.elem;
  return EDV_OK;
}

// ---- live per-launch timing (bench.py roofline) --------------------------------------------
int edv_profile(edv_ctx* ctx, int on) {
  if (!ctx) return EDV_ERR_ARG;
  ctx->prof.on = on != 0;
  return EDV_OK;
}

int edv_profile_reset(edv_ctx* ctx) {
  if (!ctx) return EDV_ERR_ARG;
  ctx->prof.used = 0;
  ctx->prof.recs.clear();
  ctx->prof_agg.clear();
  ctx->prof_names.clear();
  return EDV_OK;
}

// Wait for the recorded events and fold them into per-call-site totals.  Returns the number
// of distinct call sites (>= 0) or a negative status.
int edv_profile_collect(edv_ctx* ctx) {
  if (!ctx) return EDV_ERR_ARG;
  Profiler& pr = ctx->prof;
  if (pr.used) {
    if (cudaEventSynchronize(pr.ev[pr.used - 1]) != cudaSuccess) return set_err(ctx, EDV_ERR_CUDA, "edv_profile_collect: event sync failed");
    for (size_t i = 1; i < pr.used; ++i) {
      const ProfRec& r = pr.recs[i];
      if (r.name.empty()) continue;  // start marker of a forward
      float ms = 0.f;
      if (cudaEventElapsedTime(&ms, pr.ev[i - 1], pr.ev[i]) != cudaSuccess) continue;
      auto it = ctx->prof_agg.find(r.name);
      if (it == ctx->prof_agg.end()) {
        ctx->prof_names.push_back(r.name);
        it = ctx->prof_agg.emplace(r.name, edv_ctx::Agg()).first;
      }
      it->second.ms += ms;
      it->second.flops += r.flops;
      it->second.bytes += r.bytes;
      it->second.count += 1;
    }
  }
  pr.used = 0;
  pr.recs.clear();
  return (int)ctx->prof_names.size();
}

int edv_profile_get(edv_ctx* ctx, int index, char* name, int name_cap, double* ms, long long* count, double* flops,
                    double* bytes) {
  if (!ctx || index < 0 || index >= (int)ctx->prof_names.size() || !name || name_cap < 1) return EDV_ERR_ARG;
  const std::string& n = ctx->prof_names[index];
  const edv_ctx::Agg& a = ctx->prof_agg[n];
  snprintf(name, name_cap, "%s", n.c_str());
  if (ms) *ms = a.ms;
  if (count) *count = a.count;
  if (flops) *flops = a.flops;
  if (bytes) *bytes = a.bytes;
  return EDV_OK;
}

// ---- per-kernel entry points ----------------------------------------------------------------
static int finish(Launch& L) {
  if (!L.ok()) g_create_error = L.err;
  return L.status;
}

// One GEMM / conv with a caller-described epilogue through gemm(), the forward's own kernel selection; `kernel` receives
// the instance that ran.
int edv_op_gemm(int dtype, int engine, const edv_gemm_desc* d, char* kernel, int kernel_cap, void* stream) {
  if (kernel && kernel_cap > 0) kernel[0] = 0;
  if (!d || d->struct_bytes != (int)sizeof(edv_gemm_desc))
    return set_err(nullptr, EDV_ERR_ARG, "edv_op_gemm: struct_bytes %d, library's edv_gemm_desc has %d", d ? d->struct_bytes : -1,
                   (int)sizeof(edv_gemm_desc));
  if (dtype < EDV_F32 || dtype > EDV_F16) return set_err(nullptr, EDV_ERR_ARG, "edv_op_gemm: bad dtype %d", dtype);
  const bool tc = dtype != EDV_F32 && engine == EDV_ENGINE_TC;
  // GEGLU and the disparity head exist only in the tcgen05 epilogue: the CUDA-core forward composes them from a plain GEMM
  // plus geglu_pair_kernel / head_dot_kernel, and epi_apply would silently ignore them
  if (!tc && (d->act == ACT_GEGLU || d->act == ACT_HEAD))
    return set_err(nullptr, EDV_ERR_ARG, "edv_op_gemm: act %d needs the tensor-core engine", d->act);
  if (d->act < ACT_NONE || d->act > ACT_SIGMOID || d->map < MAP_LINEAR || d->map > MAP_PIXSHUF)
    return set_err(nullptr, EDV_ERR_ARG, "edv_op_gemm: bad act %d / map %d", d->act, d->map);
  if (!d->out || !d->A || !d->W) return set_err(nullptr, EDV_ERR_ARG, "edv_op_gemm: null A, W or out");
  if (d->M < 1 || d->N < 1 || d->K < 1) return set_err(nullptr, EDV_ERR_ARG, "edv_op_gemm: empty problem");
  if (d->conv) {
    if (d->stride != 1 && (tc || d->stride != 2)) return set_err(nullptr, EDV_ERR_ARG, "edv_op_gemm: conv stride %d", d->stride);
    if (d->F < 1 || d->H < 1 || d->Wd < 1 || d->C < 1 || d->K != 9 * d->C ||
        (long long)d->M != (long long)d->F * ((d->H - 1) / d->stride + 1) * ((d->Wd - 1) / d->stride + 1))
      return set_err(nullptr, EDV_ERR_ARG, "edv_op_gemm: conv needs K = 9*C and M = F*OH*OW");
  } else if (d->lda < d->K) {
    return set_err(nullptr, EDV_ERR_ARG, "edv_op_gemm: lda < K");
  }
  // the vector-alignment contract of load_vec / store_vec (common.cuh): leading dimensions are multiples of 8 elements
  // (the head epilogue writes one float per row and has no output pitch)
  if ((!d->conv && d->lda % 8) || (d->act != ACT_HEAD && d->ldo % 8) || (d->res1 && d->ld_res1 % 8) || (d->res2 && d->ld_res2 % 8) ||
      (d->rowbias && d->rb_ld % 8))
    return set_err(nullptr, EDV_ERR_ARG, "edv_op_gemm: leading dimensions must be multiples of 8");
  Launch L;
  L.stream = (cudaStream_t)stream;
  GemmArgs a;
  a.A = d->A; a.W = d->W; a.M = d->M; a.N = d->N; a.K = d->K; a.lda = d->lda;
  a.conv = d->conv != 0; a.F = d->F; a.H = d->H; a.Wd = d->Wd; a.C = d->C; a.stride = d->stride;
  Epi& e = a.e;
  e = epi_zero();
  e.out = d->out; e.out_relu = d->out_relu; e.bias = d->bias; e.rowbias = d->rowbias;
  e.res1 = d->res1; e.res2 = d->res2; e.head_w = d->head_w;
  e.ldo = d->ldo; e.ld_res1 = d->ld_res1; e.ld_res2 = d->ld_res2; e.rb_ld = d->rb_ld;
  e.rb_div = d->rb_div; e.rb_mod = d->rb_mod;
  e.out_f32 = d->out_f32; e.res1_f32 = d->res1_f32; e.res2_f32 = d->res2_f32;
  e.act = d->act; e.map = d->map; e.map_p = d->map_p;
  e.ps_k = d->ps_k; e.ps_h = d->ps_h; e.ps_w = d->ps_w; e.ps_c = d->ps_c;
  e.head_b = 0.f;   // the head's 1x1 bias is head_w[32], as in the forward
  e.sig_sign = d->sig_sign;
  gemm(L, dtype, engine, a);
  if (kernel && kernel_cap > 0) snprintf(kernel, kernel_cap, "%s", L.kernel.c_str());
  return finish(L);
}

// edv_op_linear on the tcgen05 kernel with its in-kernel timeline: timeline_dev receives 4 x 256 clock64 stamps (slot
// table in gemm_tc.cuh).  Diagnostic evidence (which role waits on which), not a product path.
int edv_op_linear_timeline(int dtype, const void* A, const void* W, const float* bias, void* C, int M, int N, int K, int act,
                           long long* timeline_dev, void* stream) {
  if (dtype == EDV_F32 || !timeline_dev) return EDV_ERR_ARG;
  Launch L;
  L.stream = (cudaStream_t)stream;
  if (cudaMemsetAsync(timeline_dev, 0, 4 * 256 * sizeof(long long), L.stream) != cudaSuccess) return EDV_ERR_CUDA;
  GemmArgs a;
  a.A = A; a.W = W; a.M = M; a.N = N; a.K = K; a.lda = K;
  a.e = epi_zero();
  a.e.out = C; a.e.ldo = N; a.e.bias = bias; a.e.act = act;
  a.e.tim = timeline_dev;
  gemm(L, dtype, EDV_ENGINE_TC, a);
  return finish(L);
}

int edv_op_linear_residual_ln(int dtype, const void* A, const void* W, const float* bias, float* x_inout, const float* gamma,
                              const float* beta, float eps, void* xn_out, int M, int N, int K, long long* timeline_dev, void* stream) {
  if (!A || !W || !x_inout || M < 1) return EDV_ERR_ARG;
  Launch L;
  L.stream = (cudaStream_t)stream;
  const int do_ln = (gamma && beta && xn_out) ? 1 : 0;
  if (timeline_dev && cudaMemsetAsync(timeline_dev, 0, 64 * sizeof(long long), L.stream) != cudaSuccess) return EDV_ERR_CUDA;
  gemm_ln(L, dtype, A, W, bias, x_inout, xn_out, gamma, beta, eps, M, N, K, do_ln, timeline_dev);
  return finish(L);
}

int edv_op_attention(int dtype, int engine, const void* qkv, void* out, int F, int S, int heads, void* stream) {
  Launch L;
  L.stream = (cudaStream_t)stream;
  attention(L, dtype, engine, qkv, out, F, S, heads);
  return finish(L);
}

// edv_op_attention with the in-kernel timeline of the tcgen05 kernel: timeline_dev receives 8 x 64 clock64 stamps
// (slot meanings in attention_tc.cuh); evidence for DESIGN.md's per-iteration cycle budget, not a product path.
int edv_op_attention_timeline(int dtype, const void* qkv, void* out, int F, int S, int heads, long long* timeline_dev, void* stream) {
  if (dtype == EDV_F32 || !timeline_dev) return EDV_ERR_ARG;
  Launch L;
  L.stream = (cudaStream_t)stream;
  if (cudaMemsetAsync(timeline_dev, 0, 8 * 64 * sizeof(long long), L.stream) != cudaSuccess) return EDV_ERR_CUDA;
  attention(L, dtype, EDV_ENGINE_TC, qkv, out, F, S, heads, timeline_dev);
  return finish(L);
}

int edv_op_temporal_attention(int dtype, const void* qkv, void* out, int B, int T, int hw, int C, void* stream) {
  Launch L;
  L.stream = (cudaStream_t)stream;
  temporal_attention(L, dtype, qkv, out, B, T, hw, C);
  return finish(L);
}

int edv_op_disp_head(int dtype, const void* X, const void* Wt, const float* bias, const float* head_w, float* out, int F,
                     int H1, int W1, int OH, int OW, int Cin, float sig_sign, void* stream) {
  Launch L;
  L.stream = (cudaStream_t)stream;
  head_fused(L, dtype, X, Wt, bias, head_w, out, F, H1, W1, OH, OW, Cin, sig_sign);
  return finish(L);
}

int edv_op_cubic_resize_u8(const uint8_t* src, float* dst, int N, int H, int W, int h, int w, void* stream) {
  if (!src || !dst || N < 1 || H < 1 || W < 1 || h < 1 || w < 1) return EDV_ERR_ARG;
  Launch L;
  L.stream = (cudaStream_t)stream;
  const long long total = (long long)N * h * w;
  L.note(0, (double)N * H * W * 3 + (double)total * 12);
  cubic_resize_u8_kernel<<<nblk(total, 256), 256, 0, L.stream>>>(src, dst, N, H, W, h, w);
  L.check("cubic_resize_u8");
  return finish(L);
}

int edv_op_layernorm(int dtype, const float* X, const float* gamma, const float* beta, void* Y, int M, int D,
                     float eps, void* stream) {
  Launch L;
  L.stream = (cudaStream_t)stream;
  layernorm(L, dtype, X, gamma, beta, Y, M, D, eps);
  return finish(L);
}

int edv_op_groupnorm(int dtype, const void* X, const float* gamma, const float* beta, void* Y, int F, int hw, int C,
                     float eps, void* stream) {
  Launch L;
  L.stream = (cudaStream_t)stream;
  float2* stats = nullptr;
  if (cudaMallocAsync((void**)&stats, (size_t)F * 32 * (1 + GN_MAX_SPLIT) * sizeof(float2), L.stream) != cudaSuccess) return EDV_ERR_CUDA;
  groupnorm(L, dtype, X, gamma, beta, Y, stats, F, hw, C, eps);
  cudaFreeAsync(stats, L.stream);
  return finish(L);
}

int edv_op_upsample(int dtype, const void* X, void* Y, int F, int h, int w, int oh, int ow, int C, void* stream) {
  Launch L;
  L.stream = (cudaStream_t)stream;
  upsample(L, dtype, X, Y, F, h, w, oh, ow, C);
  return finish(L);
}

int edv_op_resize_f32(const float* X, float* Y, int F, int h, int w, int oh, int ow, void* stream) {
  Launch L;
  L.stream = (cudaStream_t)stream;
  resize_f32(L, X, Y, F, h, w, oh, ow);
  return finish(L);
}

int edv_op_disp_to_depth(const float* disp_dev, float* scaled_disp_dev, float* depth_dev, long long n, double min_depth,
                         double max_depth, void* stream) {
  if (!disp_dev || !depth_dev || n < 1 || !(min_depth > 0) || !(max_depth > 0)) return EDV_ERR_ARG;
  Launch L;
  L.stream = (cudaStream_t)stream;
  const double min_disp = 1.0 / max_depth, max_disp = 1.0 / min_depth;   // Python floats in the reference
  L.note(0, (double)n * (scaled_disp_dev ? 12 : 8));
  disp_to_depth_kernel<<<nblk(n, 256), 256, 0, L.stream>>>(disp_dev, scaled_disp_dev, depth_dev, n, (float)min_disp,
                                                         (float)(max_disp - min_disp));
  L.check("disp_to_depth");
  return finish(L);
}

int edv_op_compute_errors(const float* gt_dev, const float* pred_dev, const uint8_t* mask_dev, int frames, long long hw,
                          float gt_lo, float gt_hi, float pred_scale, float clamp_lo, float clamp_hi, double* out_dev,
                          void* stream) {
  if (!gt_dev || !pred_dev || !out_dev || frames < 1 || hw < 1) return EDV_ERR_ARG;
  Launch L;
  L.stream = (cudaStream_t)stream;
  L.note(0, (double)frames * hw * (mask_dev ? 9 : 8));
  compute_errors_kernel<<<frames, CE_THREADS, 0, L.stream>>>(gt_dev, pred_dev, mask_dev, hw, gt_lo, gt_hi, pred_scale, clamp_lo,
                                                            clamp_hi, out_dev);
  L.check("compute_errors");
  return finish(L);
}

long long edv_op_stitch_plan(int H, int W, int32_t* plan_host, long long cap) {
  if (H < 1 || W < 1 || 8LL * H * W >= (1LL << 24)) return EDV_ERR_ARG;   // np.sum(ones) must stay exact in float32
  const std::vector<int> plan = stitch_plan_build(8LL * H * W);
  if (plan_host && cap >= (long long)plan.size()) memcpy(plan_host, plan.data(), plan.size() * sizeof(int));
  return (long long)plan.size();
}

int edv_op_stitch_window(const float* win_dev, int k, int H, int W, float* out_dev, const int32_t* plan_dev, int n_leaves,
                         float* scratch_dev, float* scale_shift_dev, void* stream) {
  if (!win_dev || !out_dev || !plan_dev || !scratch_dev || !scale_shift_dev || k < 0 || H < 1 || W < 1 || n_leaves < 1)
    return EDV_ERR_ARG;
  if (((uintptr_t)scratch_dev & 15) != 0) return EDV_ERR_ARG;
  Launch L;
  L.stream = (cudaStream_t)stream;
  const long long hw = (long long)H * W;
  if (k == 0) {
    // depth_list_aligned += depth_list[:INFER_LEN] (endodav.py:220-221)
    cudaError_t e = cudaMemcpyAsync(out_dev, win_dev, (size_t)32 * hw * sizeof(float), cudaMemcpyDeviceToDevice, L.stream);
    if (e != cudaSuccess) return EDV_ERR_CUDA;
    stitch_identity_kernel<<<1, 1, 0, L.stream>>>(scale_shift_dev);
    L.check("stitch_identity");
    return finish(L);
  }
  const long long pos = 32 + 22LL * (k - 1);        // frames aligned so far
  float* tail = out_dev + (pos - 8) * hw;            // depth_list_aligned[-INTERP_LEN:]
  const long long n = 8 * hw;
  float* ss = scale_shift_dev + 2 * (long long)k;
  float4* val = (float4*)scratch_dev;
  L.note(0, (double)n * 8);
  stitch_leaf_kernel<<<nblk((long long)n_leaves * 8, STITCH_THREADS), STITCH_THREADS, 0, L.stream>>>(tail, win_dev + 2 * hw, plan_dev, val);
  L.check("stitch_leaf");
  stitch_tree_solve_kernel<<<1, 1024, 0, L.stream>>>(plan_dev, val, n, ss);
  L.check("stitch_tree_solve");
  StitchFade f;
  const double step = (1.0 - 0.0) / 7;               // get_interpolate_frames (utils/util.py:65-74)
  for (int i = 0; i < 8; ++i) {
    const double w = i == 0 ? 0.0 : (i == 7 ? 1.0 : i * step);
    f.w1[i] = (float)w;
    f.w0[i] = (float)(1 - w);
  }
  L.note(0, (double)hw * (30 + 30 + 8) * 4);
  stitch_apply_kernel<<<nblk(30 * hw, 256), 256, 0, L.stream>>>(win_dev, tail, hw, ss, f);
  L.check("stitch_apply");
  return finish(L);
}

}  // extern "C"
