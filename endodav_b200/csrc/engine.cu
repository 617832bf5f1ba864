// endodav_b200 engine: context, weight registry, shape plan and the forward graph of
// endodav.forward (models/endodav/endodav.py:150-160) expressed as a fixed sequence of
// sm_100a kernel launches on the caller's stream.  C ABI in include/endodav_b200.h.
#include <cuda_runtime.h>

#include <algorithm>
#include <cfloat>
#include <climits>
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

// One workspace buffer.  `name` is empty when the plan's configuration does not need the buffer.
struct Buf {
  std::string name;
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

// scratch of one temporal module (Fwd::motion); gg2 only on the CUDA-core engine
struct MMScratch {
  Buf stats, gn, hs, ln, qkv, att, gg, hsT, gg2;
};

struct Plan {
  bool valid = false;
  int B = 0, T = 0, H = 0, W = 0, h = 0, w = 0;
  int BT = 0, ph = 0, pw = 0, P = 0, N = 0;
  long long M = 0, Mp = 0;
  int ph2 = 0, pw2 = 0;
  int Cp[4] = {0, 0, 0, 0};
  int out_h[4] = {0, 0, 0, 0}, out_w[4] = {0, 0, 0, 0};
  MMPlan mod[4];            // geometry of temporal module j
  // the path choices that decide which optional buffers exist; the forward follows them
  bool tc = false;          // tensor-core engine (else CUDA-core)
  bool fused_head = false;  // the disparity head runs as one kernel (head_fused.cuh): no head.up map
  size_t total = 0;
  // workspace buffers (edv_plan gives their layout order)
  Buf A0, x, xn, qkv, ao, hid;             // hid: the MLP's hidden activations ("h")
  Buf tap[4], tapc[4], rorb[4], tapr[4];   // final-norm taps; tapc / rorb / tapr: use_clstoken readout
  Buf rb_pt, rb_t1, rb_t2, rb_t3;          // residual bottleneck blocks
  Buf L1, L2, L3, L4p, L4, col, L3m, L4m;
  MMScratch mm, mmb;                       // mmb: module 0, which runs on the side stream beside module 1
  Buf lr[4], lrr[4];                       // layer{1-4}_rn outputs and their relu copies
  Buf ref_tmp, ref_s, ref_sr, ref_u, ref_v;
  Buf p4, p4m, p3, p3m, p2, p1;
  Buf head_o1, head_up, head_t32;
  Buf disp[4];
  struct {
    DebugTap tokens0, block0, tap[4], layer[4], mm[2], path4_pre, path3, path1;
  } dbg;                                   // debug taps (planned with edv_set_debug on)
  std::vector<Buf> bufs;                   // every planned buffer, for edv_plan_buffer
  std::vector<DebugTap> taps;              // every debug tap, for edv_debug_tap
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
  unsigned long long last_use = 0;   // graph_clock of the last replay (LRU eviction of graphs)
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
    eng = ctx->plan.tc ? EDV_ENGINE_TC : EDV_ENGINE_SIMT;
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

  void* at(const Buf& b) {
    if (b.name.empty()) {
      L.fail(EDV_ERR_STATE, "internal: the forward reached a workspace buffer that its plan did not create");
      return nullptr;
    }
    return ws + b.off;
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
  // debug tap t <- the first t.cols channels of t.rows rows of src (row pitch ld_src elements)
  void snapshot(const DebugTap& t, const void* src, int ld_src, bool src_f32) {
    if (!c->debug || !L.ok()) return;
    float* dst = (float*)at(t.buf);
    if (!dst) return;
    long long n = t.rows * t.cols;
    if (src_f32) copy_channels_f32_kernel<float><<<nblk(n, 256), 256, 0, L.stream>>>((const float*)src, dst, t.rows, ld_src, t.cols);
    else EDV_DISPATCH_T(dt, { copy_channels_f32_kernel<T><<<nblk(n, 256), 256, 0, L.stream>>>((const T*)src, dst, t.rows, ld_src, t.cols); });
    L.check("debug snapshot");
  }

  // TemporalModule (motion_module.py:60-65,102-126,164-177): X [BT*hw, C] NHWC -> Y same
  // `s`: scratch family (mm on the main stream, mmb for the module that runs beside it on the side stream)
  void motion(int j, const void* X, void* Y, const MMScratch& s) {
    const Plan& p = c->plan;
    const int C = p.mod[j].C, hw = p.mod[j].h * p.mod[j].w, T = p.T, B = p.B;
    const long long Mm = (long long)p.BT * hw;
    const std::string n = "mm" + std::to_string(j) + ".";
    void* gnb = at(s.gn);
    float* hs = (float*)at(s.hs);
    void* lnb = at(s.ln);
    void* qkvb = at(s.qkv);
    void* att = at(s.att);
    void* gg = at(s.gg);
    void* hsT = at(s.hsT);
    groupnorm(L, dt, X, wf(n + "gn.w", C), wf(n + "gn.b", C), gnb, (float2*)at(s.stats), p.BT, hw, C, 1e-6f);
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
      void* tmp = at(s.gg2);
      linear(lnb, Mm, C, n + "geglu.w", 8 * C, ep(tmp, 8 * C, wf(n + "geglu.b", 8 * C)));
      geglu_pair(L, dt, tmp, gg, Mm, 4 * C);
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
    void* tmp = at(p.ref_tmp);
    void* s = at(p.ref_s);
    void* sr = at(p.ref_sr);
    void* u = at(p.ref_u);
    void* v = at(p.ref_v);
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
    void* o1 = at(p.head_o1);
    conv3(X, p.BT, H, Wd, F_, c0 + ".w", Fh, ep(o1, Fh, wf(c0 + ".b", Fh)));
    const float* hw_ = wf(c4 + ".w", 33);
    if (p.fused_head) {
      // K14: the upsampled map and the 32-channel conv output never touch HBM
      L.tag = tag_of(c2);
      head_fused(L, dt, o1, wt(c2 + ".w", (size_t)32 * 9 * Fh), wf(c2 + ".b", 32), hw_, out, p.BT, H, Wd, OH, OW, Fh, sig_sign);
      L.tag.clear();
      return;
    }
    void* up = at(p.head_up);
    upsample(L, dt, o1, up, p.BT, H, Wd, OH, OW, Fh);
    if (tc()) {
      Epi e = ep(out, 1, wf(c2 + ".b", 32));
      e.act = ACT_HEAD; e.head_w = hw_; e.sig_sign = sig_sign; e.out_f32 = 1;
      e.head_b = 0.f;  // the kernel adds head_w[32]
      conv3(up, p.BT, OH, OW, Fh, c2 + ".w", 32, e);
    } else {
      void* t32 = at(p.head_t32);
      Epi e = ep(t32, 32, wf(c2 + ".b", 32));
      e.act = ACT_RELU;
      conv3(up, p.BT, OH, OW, Fh, c2 + ".w", 32, e);
      head_dot(L, dt, t32, hw_, out, (long long)p.BT * OH * OW, 32, sig_sign);
    }
  }

  int run(const void* frames, bool u8, float* const disp[4], float* resized, int out_h, int out_w) {
    const Plan& p = c->plan;
    const edv_config& g = c->cfg;
    const int D = g.dim;
    L.begin();
    // ---- K1 + K2: preprocess, patch embedding (patch_embed.py:75-77; vision_transformer.py:219-227)
    void* A0 = at(p.A0);
    float* x = (float*)at(p.x);
    {
      // endodac with pre_norm=False feeds raw [0,1] pixels (endodac.py:208-211)
      preprocess_patches(L, dt, frames, u8, A0, p.BT, p.H, p.W, p.h, p.w, KPATCH, g.no_normalize ? 0 : 1);
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
    snapshot(p.dbg.tokens0, x, D, true);
    // ---- encoder blocks (block.py:110-151)
    void* xn = at(p.xn);
    void* qkv = at(p.qkv);
    void* ao = at(p.ao);
    void* hb = at(p.hid);
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
      if (i == 0) snapshot(p.dbg.block0, x, D, true);
      if (tap_i < 4 && i == g.taps[tap_i]) {
        void* tap = at(p.tap[tap_i]);
        // final norm on the tap + cls split (vision_transformer.py:318-321)
        layernorm(L, dt, x, wf("norm.w", D), wf("norm.b", D), tap, p.Mp, D, 1e-6f, g.no_cls ? 0 : p.N, g.no_cls ? 0 : 1);
        snapshot(p.dbg.tap[tap_i], tap, D, false);
        if (g.use_clstoken) {
          // readout projects (dpt.py:92-99; dpt_pyramid.py:54-57): tap' = GELU(Linear(2D, D)([token | class token])) =
          // GELU(token W1^T + rb[frame]) with the per-frame row bias rb = class token W2^T + b.  The class token is row 0
          // of the frame after the final norm (without a cls token: its first patch token, as in the reference).
          void* cls_tok = at(p.tapc[tap_i]);
          float* rb = (float*)at(p.rorb[tap_i]);
          const std::string ro = "ro" + std::to_string(tap_i) + ".";
          layernorm(L, dt, x, wf("norm.w", D), wf("norm.b", D), cls_tok, p.BT, D, 1e-6f, p.N, -1);
          {
            Epi e = ep(rb, D, wf(ro + "b", D));
            e.out_f32 = 1;
            linear(cls_tok, p.BT, D, ro + "w2", D, e);
          }
          {
            Epi e = ep(at(p.tapr[tap_i]), D, nullptr);
            e.rowbias = rb;
            e.rb_div = p.P; e.rb_mod = p.BT; e.rb_ld = D;
            e.act = ACT_GELU;
            linear(tap, p.Mp, D, ro + "w1", D, e);
          }
        }
        ++tap_i;
      }
    }
    if (tap_i != 4) L.fail(EDV_ERR_ARG, "taps must be increasing block indices < depth");
    // ---- DPT head (dpt_pyramid.py:51-113)
    const int F_ = g.features;
    void* L1 = at(p.L1);
    void* L2 = at(p.L2);
    void* L3 = at(p.L3);
    void* L4p = at(p.L4p);
    void* L4 = at(p.L4);
    // endodac (models/endodac/endodac.py:93-127) is this head without the four temporal modules
    const bool mm_on = !g.no_motion;
    void* L3m = mm_on ? at(p.L3m) : L3;
    void* L4m = mm_on ? at(p.L4m) : L4;
    void *l1r = at(p.lr[0]), *l2r = at(p.lr[1]), *l3r = at(p.lr[2]), *l4r = at(p.lr[3]);
    void *l1rr = at(p.lrr[0]), *l2rr = at(p.lrr[1]), *l3rr = at(p.lrr[2]), *l4rr = at(p.lrr[3]);
    const Buf* tap_out = g.use_clstoken ? p.tapr : p.tap;   // what the reassemble projections read
    // The decoder is a DAG: paths 1-3 (reassemble -> [temporal module 0] -> layer_rn) only meet the deep path at
    // their fusion blocks.  The deep path (path 4 -> refinenet4 -> module 2 -> refinenet3 -> module 3 -> ...) is a
    // chain of small, latency-bound launches on 19 x 19 / 37 x 37 maps that leaves most SMs idle, so paths 1-3 run
    // beside it on the side stream (same kernels, same buffers per tensor: bit-identical to the serial order).
    fork_side();
    {
      // projects[0] (1x1) merged with resize_layers[0] (ConvT k4 s4): one GEMM + pixel shuffle
      Epi e = ep(L1, p.Cp[0], wf("proj0.b", 16 * p.Cp[0]));
      e.map = MAP_PIXSHUF; e.ps_k = 4; e.ps_h = p.ph; e.ps_w = p.pw; e.ps_c = p.Cp[0];
      linear(at(tap_out[0]), p.Mp, D, "proj0.w", 16 * p.Cp[0], e);
    }
    {
      Epi e = ep(L2, p.Cp[1], wf("proj1.b", 4 * p.Cp[1]));
      e.map = MAP_PIXSHUF; e.ps_k = 2; e.ps_h = p.ph; e.ps_w = p.pw; e.ps_c = p.Cp[1];
      linear(at(tap_out[1]), p.Mp, D, "proj1.w", 4 * p.Cp[1], e);
    }
    linear(at(tap_out[2]), p.Mp, D, "proj2.w", p.Cp[2], ep(L3, p.Cp[2], wf("proj2.b", p.Cp[2])));
    if (mm_on) motion(0, L3, L3m, par ? p.mmb : p.mm);
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
    linear(at(tap_out[3]), p.Mp, D, "proj3.w", p.Cp[3], ep(L4p, p.Cp[3], wf("proj3.b", p.Cp[3])));
    {
      // resize_layers[3]: 3x3 stride 2 pad 1 (dpt.py:85-90) = explicit im2col + GEMM
      const long long Mo = (long long)p.BT * p.ph2 * p.pw2;
      if (tc()) {
        void* col = at(p.col);
        im2col3x3(L, dt, L4p, col, p.BT, p.ph, p.pw, p.Cp[3], p.ph2, p.pw2, 2);
        linear(col, Mo, 9 * p.Cp[3], "resize3.w", p.Cp[3], ep(L4, p.Cp[3], wf("resize3.b", p.Cp[3])));
      } else {
        GemmArgs a;
        a.A = L4p; a.W = wt("resize3.w", (size_t)p.Cp[3] * 9 * p.Cp[3]); a.M = (int)Mo; a.N = p.Cp[3]; a.K = 9 * p.Cp[3];
        a.e = ep(L4, p.Cp[3], wf("resize3.b", p.Cp[3]));
        a.conv = true; a.F = p.BT; a.H = p.ph; a.Wd = p.pw; a.C = p.Cp[3]; a.stride = 2;
        if (L.ok()) gemm(L, dt, eng, a);
      }
    }
    if (mm_on) motion(1, L4, L4m, p.mm);
    {
      Epi e = ep(l4r, F_, nullptr); e.out_relu = l4rr;
      conv3(L4m, p.BT, p.ph2, p.pw2, p.Cp[3], "rn4.w", F_, e);
    }
    snapshot(p.dbg.layer[0], L1, p.Cp[0], false);
    snapshot(p.dbg.layer[1], L2, p.Cp[1], false);
    snapshot(p.dbg.layer[2], L3, p.Cp[2], false);
    snapshot(p.dbg.layer[3], L4, p.Cp[3], false);
    snapshot(p.dbg.mm[0], L3m, p.Cp[2], false);
    snapshot(p.dbg.mm[1], L4m, p.Cp[3], false);
    void *p4 = at(p.p4), *p3 = at(p.p3), *p2 = at(p.p2), *p1 = at(p.p1);
    void *p4m = mm_on ? at(p.p4m) : p4, *p3m = mm_on ? at(p.p3m) : p3;
    fusion(4, l4r, l4rr, nullptr, nullptr, p.ph2, p.pw2, p.ph, p.pw, p4);
    snapshot(p.dbg.path4_pre, p4, F_, false);
    if (mm_on) motion(2, p4, p4m, p.mm);
    join_side();   // refinenet3 is the first consumer of the side stream's layer{1,2,3}_rn maps
    fusion(3, p4m, nullptr, l3r, l3rr, p.ph, p.pw, 2 * p.ph, 2 * p.pw, p3);
    if (mm_on) motion(3, p3, p3m, p.mm);
    snapshot(p.dbg.path3, p3m, F_, false);
    fusion(2, p3m, nullptr, l2r, l2rr, 2 * p.ph, 2 * p.pw, 4 * p.ph, 4 * p.pw, p2);
    fusion(1, p2, nullptr, l1r, l1rr, 4 * p.ph, 4 * p.pw, 8 * p.ph, 8 * p.pw, p1);
    snapshot(p.dbg.path1, p1, F_, false);
    // ---- disparity outputs
    float* d[4];
    for (int s = 0; s < 4; ++s) d[s] = disp[s] ? disp[s] : (float*)at(p.disp[s]);
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
    void* pt = at(p.rb_pt);
    void* t1 = at(p.rb_t1);
    void* t2 = at(p.rb_t2);
    void* t3 = at(p.rb_t3);
    const int cls = c->cfg.no_cls ? 0 : 1;
    tokens_to_patches(L, dt, x, pt, p.Mp, p.P, D, cls);
    linear(pt, p.Mp, D, n + "res.c1.w", bcp, ep(t1, bcp, nullptr));
    rowln_act(L, dt, t1, wf(n + "res.n1.w", bcp), wf(n + "res.n1.b", bcp), t2, p.Mp, bcp, bc, 1e-6f, 1, "res ln1");
    conv3(t2, p.BT, p.ph, p.pw, bcp, n + "res.c2.w", bcp, ep(t1, bcp, nullptr));
    rowln_act(L, dt, t1, wf(n + "res.n2.w", bcp), wf(n + "res.n2.b", bcp), t2, p.Mp, bcp, bc, 1e-6f, 1, "res ln2");
    linear(t2, p.Mp, bcp, n + "res.c3.w", D, ep(t3, D, nullptr));
    resblock_add(L, dt, x, t3, wf(n + "res.n3.w", D), wf(n + "res.n3.b", D), p.Mp, p.P, D, 1e-6f, cls);
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
  p.mod[0] = MMPlan{p.Cp[2], p.ph, p.pw};
  p.mod[1] = MMPlan{p.Cp[3], p.ph2, p.pw2};
  p.mod[2] = MMPlan{F_, p.ph, p.pw};
  p.mod[3] = MMPlan{F_, 2 * p.ph, 2 * p.pw};
  for (int j = 0; j < 4 && !g.no_motion; ++j) {
    int hd = p.mod[j].C / 8;
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

  p.tc = g.dtype != EDV_F32 && g.engine != EDV_ENGINE_SIMT;
  p.fused_head = p.tc && head_fused_supported(g.dtype, Fh);

  // Workspace layout: each buffer is placed here, in this order, at a 1 KiB-aligned offset.
  const int es = (int)dtype_size(g.dtype);
  size_t off = 0;
  auto place = [&](Buf& b, std::string name, size_t count, int elem) {
    b.name = std::move(name);
    b.off = off;
    b.bytes = count * elem;
    b.elem = elem;
    off += (b.bytes + 1023) & ~(size_t)1023;
  };
  auto add = [&](Buf& b, std::string name, size_t count, int elem) {
    place(b, std::move(name), count, elem);
    p.bufs.push_back(b);
  };
  const int D = g.dim;
  add(p.A0, "A0", (size_t)p.Mp * KPATCH, es);
  add(p.x, "x", (size_t)p.M * D, 4);
  add(p.xn, "xn", (size_t)p.M * D, es);
  add(p.qkv, "qkv", (size_t)p.M * 3 * D, es);
  add(p.ao, "ao", (size_t)p.M * D, es);
  add(p.hid, "h", (size_t)p.M * 4 * D, es);
  for (int i = 0; i < 4; ++i) {
    const std::string n = std::to_string(i);
    add(p.tap[i], "tap" + n, (size_t)p.Mp * D, es);
    if (g.use_clstoken) {
      add(p.tapc[i], "tapc" + n, (size_t)p.BT * D, es);
      add(p.rorb[i], "rorb" + n, (size_t)p.BT * D, 4);
      add(p.tapr[i], "tapr" + n, (size_t)p.Mp * D, es);
    }
  }
  if (g.res_blocks) {
    const int bcp = round_up(D / 8, 64);
    add(p.rb_pt, "rb.pt", (size_t)p.Mp * D, es);
    add(p.rb_t1, "rb.t1", (size_t)p.Mp * bcp, es);
    add(p.rb_t2, "rb.t2", (size_t)p.Mp * bcp, es);
    add(p.rb_t3, "rb.t3", (size_t)p.Mp * D, es);
  }
  const size_t px1 = (size_t)p.BT * 16 * p.P, px2 = (size_t)p.BT * 4 * p.P, px3 = (size_t)p.Mp, px4 = (size_t)p.BT * p.ph2 * p.pw2;
  const size_t px0 = (size_t)p.BT * 64 * p.P;  // 8ph x 8pw
  const size_t px[4] = {px1, px2, px3, px4};   // layer{1-4}
  add(p.L1, "L1", px1 * p.Cp[0], es);
  add(p.L2, "L2", px2 * p.Cp[1], es);
  add(p.L3, "L3", px3 * p.Cp[2], es);
  add(p.L4p, "L4p", px3 * p.Cp[3], es);
  add(p.L4, "L4", px4 * p.Cp[3], es);
  if (p.tc) add(p.col, "col", px4 * 9 * p.Cp[3], es);
  if (!g.no_motion) {
    add(p.L3m, "L3m", px3 * p.Cp[2], es);
    add(p.L4m, "L4m", px4 * p.Cp[3], es);
    // temporal-module scratch: mm sized for the largest of the four modules, mmb for module 0
    size_t mmC = 0;
    for (int j = 0; j < 4; ++j) mmC = std::max(mmC, (size_t)p.BT * p.mod[j].h * p.mod[j].w * p.mod[j].C);
    const size_t r0 = (size_t)p.BT * p.mod[0].h * p.mod[0].w * p.mod[0].C;
    auto add_mm = [&](MMScratch& s, const std::string& set, size_t n) {
      add(s.stats, set + "stats", (size_t)p.BT * 32 * (1 + GN_MAX_SPLIT), (int)sizeof(float2));
      add(s.gn, set + "gn", n, es);
      add(s.hs, set + "hs", n, 4);
      add(s.ln, set + "ln", n, es);
      add(s.qkv, set + "qkv", 3 * n, es);
      add(s.att, set + "att", n, es);
      add(s.gg, set + "gg", 4 * n, es);
      add(s.hsT, set + "hsT", n, es);
    };
    add_mm(p.mm, "mm.", mmC);
    add_mm(p.mmb, "mmb.", r0);
    if (!p.tc) {
      add(p.mm.gg2, "mm.gg2", 8 * mmC, es);
      add(p.mmb.gg2, "mmb.gg2", 8 * r0, es);
    }
  }
  for (int i = 0; i < 4; ++i) {
    const std::string n = "l" + std::to_string(i + 1);
    add(p.lr[i], n + "r", px[i] * F_, es);
    add(p.lrr[i], n + "rr", px[i] * F_, es);
  }
  // refinenet scratch at the largest input resolution (refinenet1 runs at 4ph x 4pw)
  add(p.ref_tmp, "ref.tmp", px1 * F_, es);
  add(p.ref_s, "ref.s", px1 * F_, es);
  add(p.ref_sr, "ref.sr", px1 * F_, es);
  add(p.ref_u, "ref.u", px1 * F_, es);
  add(p.ref_v, "ref.v", px1 * F_, es);
  add(p.p4, "p4", px3 * F_, es);
  add(p.p4m, "p4m", px3 * F_, es);
  add(p.p3, "p3", px2 * F_, es);
  add(p.p3m, "p3m", px2 * F_, es);
  add(p.p2, "p2", px1 * F_, es);
  add(p.p1, "p1", px0 * F_, es);
  // disparity head scratch: conv at up to 8ph x 8pw, upsample target up to out_h[0] x out_w[0]
  const size_t pxo = (size_t)p.BT * p.out_h[0] * p.out_w[0];
  add(p.head_o1, "head.o1", px0 * Fh, es);
  if (!p.fused_head) add(p.head_up, "head.up", pxo * Fh, es);
  if (!p.tc) add(p.head_t32, "head.t32", pxo * 32, es);
  for (int s = 0; s < 4; ++s) add(p.disp[s], "disp" + std::to_string(s), (size_t)p.BT * p.out_h[s] * p.out_w[s], 4);
  if (ctx->debug) {
    auto tap = [&](DebugTap& t, std::string name, long long rows, int cols) {
      place(t.buf, std::move(name), (size_t)rows * cols, 4);
      t.rows = rows;
      t.cols = cols;
      p.taps.push_back(t);
    };
    tap(p.dbg.tokens0, "tokens0", p.M, D);
    tap(p.dbg.block0, "block0", p.M, D);
    for (int i = 0; i < 4; ++i) tap(p.dbg.tap[i], "tap" + std::to_string(i), p.Mp, D);
    for (int i = 0; i < 4; ++i) tap(p.dbg.layer[i], "layer" + std::to_string(i + 1), px[i], g.out_channels[i]);
    tap(p.dbg.mm[0], "mm0", px3, g.out_channels[2]);
    tap(p.dbg.mm[1], "mm1", px4, g.out_channels[3]);
    tap(p.dbg.path4_pre, "path4_pre", px3, F_);
    tap(p.dbg.path3, "path3", px2, F_);
    tap(p.dbg.path1, "path1", px0, F_);
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
  PyramidCopy c;
  c.start[0] = 0;
  bool vec = true, any = false;
  size_t bytes[4];
  const unsigned char* src[4];
  for (int s = 0; s < 4; ++s) {
    c.src[s] = nullptr; c.dst[s] = nullptr; c.n4[s] = 0; bytes[s] = 0; src[s] = nullptr;
    if (disp[s]) {
      const size_t n = (size_t)ctx->plan.BT * ctx->plan.out_h[s] * ctx->plan.out_w[s];
      bytes[s] = n * sizeof(float);
      src[s] = (const unsigned char*)workspace_dev + ctx->plan.disp[s].off;
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

// Capture the forward on the private capture stream into key.exec / key.launches.  False when that gave no graph
// (graph_note says why): the caller then runs the forward eagerly.
static bool capture(edv_ctx* ctx, GraphEntry& key, const void* frames, bool u8, float* resized_dev, int out_h, int out_w,
                    void* workspace_dev) {
  // Capture on a private stream and replay on the caller's: the capture itself executes nothing, and the caller's
  // stream is usually torch's current stream = the legacy default stream, which cudaStreamBeginCapture refuses.
  int prio_lo = 0, prio_hi = 0;
  cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);   // the captured main chain outranks the side-stream branches
  if (!ctx->cap_stream && cudaStreamCreateWithPriority(&ctx->cap_stream, cudaStreamNonBlocking, prio_hi) != cudaSuccess) {
    ctx->graph_note = std::string("cudaStreamCreateWithPriority: ") + cudaGetErrorString(cudaGetLastError());
    ctx->cap_stream = nullptr;
    ctx->graph_mode = 0;
    return false;
  }
  cudaStream_t cap = ctx->cap_stream;
  cudaError_t be = cudaStreamBeginCapture(cap, cudaStreamCaptureModeThreadLocal);
  if (be != cudaSuccess) {
    ctx->graph_note = std::string("cudaStreamBeginCapture: ") + cudaGetErrorString(be);
    cudaGetLastError();
    return false;
  }
  int rc;
  {
    float* none[4] = {nullptr, nullptr, nullptr, nullptr};
    Fwd f(ctx, workspace_dev, cap);
    rc = f.run(frames, u8, none, resized_dev, out_h, out_w);   // pyramid into the plan's own buffers (see GraphEntry)
    key.launches = f.L.count;
  }
  cudaGraph_t graph = nullptr;
  const cudaError_t ce = cudaStreamEndCapture(cap, &graph);
  if (rc != EDV_OK || ce != cudaSuccess || !graph) {
    if (graph) cudaGraphDestroy(graph);
    ctx->graph_note = rc != EDV_OK ? std::string("forward failed under capture: ") + ctx->err : std::string("cudaStreamEndCapture: ") + cudaGetErrorString(ce);
    cudaGetLastError();
    ctx->graph_mode = 0;   // capture is not possible in this process: stay eager (and say why in edv_graph_status)
    return false;
  }
  const cudaError_t ie = cudaGraphInstantiate(&key.exec, graph, 0);
  cudaGraphDestroy(graph);
  if (ie != cudaSuccess || !key.exec) {
    ctx->graph_note = std::string("cudaGraphInstantiate: ") + cudaGetErrorString(ie);
    cudaGetLastError();
    ctx->graph_mode = 0;
    return false;
  }
  ctx->graph_note = "ok";
  return true;
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
  auto eager = [&] {
    Fwd f(ctx, workspace_dev, st);
    return f.run(frames, u8, disp, resized_dev, out_h, out_w);
  };
  auto replay = [&](const GraphEntry& g) {
    ctx->last_launches = g.launches;
    if (cudaGraphLaunch(g.exec, st) != cudaSuccess) return set_err(ctx, EDV_ERR_CUDA, "edv_forward: cudaGraphLaunch failed: %s", cudaGetErrorString(cudaGetLastError()));
    return copy_pyramid_out(ctx, disp, workspace_dev, st);
  };
  const bool graphable = ctx->graph_mode && !ctx->prof.on && !ctx->debug && ctx->plan_warm;
  if (!graphable) {
    const int rc = eager();
    if (rc == EDV_OK) ctx->plan_warm = true;
    return rc;
  }
  GraphEntry key;
  key.frames = frames; key.resized = resized_dev; key.workspace = workspace_dev;
  key.u8 = u8; key.out_h = resized_dev ? out_h : 0; key.out_w = resized_dev ? out_w : 0;
  ++ctx->graph_clock;
  for (GraphEntry& g : ctx->graphs)
    if (g.same(key)) {
      g.last_use = ctx->graph_clock;
      return replay(g);
    }
  // A capture costs about as much as a forward at the reference's resolution, so a pointer set is captured only the
  // SECOND time it comes by: a caller whose buffers never repeat (fresh tensors from a cold or fragmented allocator,
  // outputs pinned by record_stream) runs eagerly and pays nothing, a steady caller replays from its third call on.
  auto met = std::find_if(ctx->seen.begin(), ctx->seen.end(), [&](const GraphEntry& g) { return g.same(key); });
  if (met == ctx->seen.end()) {
    if (ctx->seen.size() >= 4 * (size_t)edv_ctx::GRAPH_SLOTS) ctx->seen.erase(ctx->seen.begin());
    ctx->seen.push_back(key);
    return eager();
  }
  *met = ctx->seen.back();
  ctx->seen.pop_back();
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(st, &cs) != cudaSuccess || cs != cudaStreamCaptureStatusNone) {
    // the caller is capturing this stream itself: just record our launches into its graph
    cudaGetLastError();
    return eager();
  }
  if (!capture(ctx, key, frames, u8, resized_dev, out_h, out_w, workspace_dev)) return eager();
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
  return replay(key);
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
  for (const DebugTap& t : ctx->plan.taps)
    if (t.buf.name == name) {
      *offset_bytes = t.buf.off;
      *rows = t.rows;
      *cols = t.cols;
      return EDV_OK;
    }
  return set_err(ctx, EDV_ERR_ARG, "edv_debug_tap: unknown tap '%s'", name);
}

// Enumerate the named workspace buffers of the current plan (range / saturation checks of the 16-bit
// intermediates: the Python host views its own workspace tensor at `offset_bytes`).  Returns EDV_ERR_ARG
// past the last buffer.
int edv_plan_buffer(edv_ctx* ctx, int index, char* name, int name_cap, size_t* offset_bytes, size_t* bytes, int* elem_bytes) {
  if (!ctx || !ctx->plan.valid || index < 0 || !name || name_cap < 1 || !offset_bytes || !bytes || !elem_bytes) return EDV_ERR_ARG;
  if (index >= (int)ctx->plan.bufs.size()) return EDV_ERR_ARG;
  const Buf& b = ctx->plan.bufs[index];
  snprintf(name, name_cap, "%s", b.name.c_str());
  *offset_bytes = b.off;
  *bytes = b.bytes;
  *elem_bytes = b.elem;
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
static bool aligned16(const void* p) { return ((uintptr_t)p & 15) == 0; }   // NULL passes: nullable pointers are checked apart

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
                              const float* beta, float eps, void* xn_out, int M, int N, int K, long long* timeline_dev, char* kernel,
                              int kernel_cap, void* stream) {
  if (kernel && kernel_cap > 0) kernel[0] = 0;
  if (dtype != EDV_BF16 && dtype != EDV_F16)
    return set_err(nullptr, EDV_ERR_ARG, "edv_op_linear_residual_ln: bad dtype %d (bf16 or f16)", dtype);
  if (!A || !W || !x_inout) return set_err(nullptr, EDV_ERR_ARG, "edv_op_linear_residual_ln: null A, W or x");
  // A, W, x and xn are the base addresses of TMA tensor maps
  if (!aligned16(A) || !aligned16(W) || !aligned16(x_inout) || !aligned16(xn_out))
    return set_err(nullptr, EDV_ERR_ARG, "edv_op_linear_residual_ln: A, W, x and xn must be 16-byte aligned");
  // a partial set would silently skip the LayerNorm (or normalise into nothing)
  const int do_ln = (gamma && beta && xn_out) ? 1 : 0;
  if (!do_ln && (gamma || beta || xn_out))
    return set_err(nullptr, EDV_ERR_ARG, "edv_op_linear_residual_ln: gamma, beta and xn must be all set or all NULL");
  // the kernel counts tiles as (M + 127) / 128 in int
  if (M < 1 || M > INT_MAX - 127) return set_err(nullptr, EDV_ERR_ARG, "edv_op_linear_residual_ln: M %d out of range", M);
  if (N != 384) return set_err(nullptr, EDV_ERR_ARG, "edv_op_linear_residual_ln: N %d (384 only)", N);
  if (K < 64 || K % 64) return set_err(nullptr, EDV_ERR_ARG, "edv_op_linear_residual_ln: K %d (a positive multiple of 64)", K);
  if (!(eps >= 0.f && eps <= FLT_MAX)) return set_err(nullptr, EDV_ERR_ARG, "edv_op_linear_residual_ln: eps must be finite and >= 0");
  Launch L;
  L.stream = (cudaStream_t)stream;
  if (timeline_dev && cudaMemsetAsync(timeline_dev, 0, 64 * sizeof(long long), L.stream) != cudaSuccess) return EDV_ERR_CUDA;
  gemm_ln(L, dtype, A, W, bias, x_inout, xn_out, gamma, beta, eps, M, N, K, do_ln, timeline_dev);
  if (kernel && kernel_cap > 0) snprintf(kernel, kernel_cap, "%s", L.kernel.c_str());
  return finish(L);
}

int edv_op_attention(int dtype, int engine, const void* qkv, void* out, int F, int S, int heads, char* kernel, int kernel_cap,
                     void* stream) {
  if (kernel && kernel_cap > 0) kernel[0] = 0;
  if (dtype < EDV_F32 || dtype > EDV_F16) return set_err(nullptr, EDV_ERR_ARG, "edv_op_attention: bad dtype %d", dtype);
  if (engine != EDV_ENGINE_TC && engine != EDV_ENGINE_SIMT) return set_err(nullptr, EDV_ERR_ARG, "edv_op_attention: bad engine %d", engine);
  if (!qkv || !out) return set_err(nullptr, EDV_ERR_ARG, "edv_op_attention: null qkv or out");
  if (F < 1 || S < 1 || heads < 1) return set_err(nullptr, EDV_ERR_ARG, "edv_op_attention: F, S and heads must be at least 1");
  // the tensor map's base address (TMA) and the 16-byte vector loads / stores of both kernels
  if (!aligned16(qkv) || !aligned16(out)) return set_err(nullptr, EDV_ERR_ARG, "edv_op_attention: qkv and out must be 16-byte aligned");
  Launch L;
  L.stream = (cudaStream_t)stream;
  attention(L, dtype, engine, qkv, out, F, S, heads);
  if (kernel && kernel_cap > 0) snprintf(kernel, kernel_cap, "%s", L.kernel.c_str());
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

int edv_op_temporal_attention(int dtype, const void* qkv, void* out, int B, int T, int hw, int C, const float* rope, char* kernel,
                              int kernel_cap, void* stream) {
  if (kernel && kernel_cap > 0) kernel[0] = 0;
  if (dtype < EDV_F32 || dtype > EDV_F16) return set_err(nullptr, EDV_ERR_ARG, "edv_op_temporal_attention: bad dtype %d", dtype);
  if (!qkv || !out) return set_err(nullptr, EDV_ERR_ARG, "edv_op_temporal_attention: null qkv or out");
  if (B < 1 || hw < 1) return set_err(nullptr, EDV_ERR_ARG, "edv_op_temporal_attention: empty problem");
  if (!aligned16(qkv) || !aligned16(out) || !aligned16(rope))
    return set_err(nullptr, EDV_ERR_ARG, "edv_op_temporal_attention: qkv, out and rope must be 16-byte aligned");
  Launch L;
  L.stream = (cudaStream_t)stream;
  temporal_attention(L, dtype, qkv, out, B, T, hw, C, rope);
  if (kernel && kernel_cap > 0) snprintf(kernel, kernel_cap, "%s", L.kernel.c_str());
  return finish(L);
}

int edv_op_disp_head(int dtype, const void* X, const void* Wt, const float* bias, const float* head_w, float* out, int F,
                     int H1, int W1, int OH, int OW, int Cin, float sig_sign, char* kernel, int kernel_cap, void* stream) {
  if (kernel && kernel_cap > 0) kernel[0] = 0;
  if (dtype != EDV_BF16 && dtype != EDV_F16) return set_err(nullptr, EDV_ERR_ARG, "edv_op_disp_head: bad dtype %d (bf16 or f16)", dtype);
  if (!X || !Wt || !bias || !head_w || !out) return set_err(nullptr, EDV_ERR_ARG, "edv_op_disp_head: null X, Wt, bias, head_w or out");
  // the producers and the weight staging read X and Wt with 16-byte vector loads
  if (!aligned16(X) || !aligned16(Wt)) return set_err(nullptr, EDV_ERR_ARG, "edv_op_disp_head: X and Wt must be 16-byte aligned");
  if (Cin != 32 && Cin != 128) return set_err(nullptr, EDV_ERR_ARG, "edv_op_disp_head: Cin %d (32 or 128)", Cin);
  // H1 or W1 = 0 would clamp the source row / column to -1 and read before X
  if (F < 1 || H1 < 1 || W1 < 1 || OH < 1 || OW < 1)
    return set_err(nullptr, EDV_ERR_ARG, "edv_op_disp_head: F, H1, W1, OH and OW must be at least 1");
  Launch L;
  L.stream = (cudaStream_t)stream;
  head_fused(L, dtype, X, Wt, bias, head_w, out, F, H1, W1, OH, OW, Cin, sig_sign);
  if (kernel && kernel_cap > 0) snprintf(kernel, kernel_cap, "%s", L.kernel.c_str());
  return finish(L);
}

// Both cubic-resize entry points: index == nullptr is the identity in one launch; a table goes out in launches of at
// most FrameTable::kMax output frames.  The arguments are validated by the callers.
static void cubic_resize_u8(Launch& L, const uint8_t* src, int H, int W, long long sn, long long sy, long long sx,
                            long long sc, const int64_t* index, int n, float* dst, int h, int w) {
  const int per = index ? FrameTable::kMax : n;
  for (int f0 = 0; f0 < n; f0 += per) {
    const int cnt = std::min(per, n - f0);
    FrameTable t = {};
    if (index) {
      t.count = cnt;
      for (int i = 0; i < cnt; ++i) t.src[i] = (int)index[f0 + i];
    }
    const long long total = (long long)cnt * h * w;
    L.note(0, (double)cnt * H * W * 3 + (double)total * 12);
    cubic_resize_u8_kernel<<<nblk(total, 256), 256, 0, L.stream>>>(src, dst + (size_t)f0 * 3 * h * w, cnt, H, W, h, w, sn,
                                                                   sy, sx, sc, t);
    L.check("cubic_resize_u8");
  }
}

int edv_op_cubic_resize_u8(const uint8_t* src, float* dst, int N, int H, int W, int h, int w, void* stream) {
  if (!src || !dst || N < 1 || H < 1 || W < 1 || h < 1 || w < 1) return EDV_ERR_ARG;
  Launch L;
  L.stream = (cudaStream_t)stream;
  cubic_resize_u8(L, src, H, W, (long long)H * W * 3, (long long)W * 3, 3, 1, nullptr, N, dst, h, w);
  return finish(L);
}

int edv_op_cubic_resize_u8_gather(const uint8_t* src, int n_src, int H, int W, long long stride_n, long long stride_y,
                                  long long stride_x, long long stride_c, const int64_t* index_host, int n, float* dst, int h,
                                  int w, void* stream) {
  const char* fn = "edv_op_cubic_resize_u8_gather";
  if (!src || !index_host || !dst) return set_err(nullptr, EDV_ERR_ARG, "%s: null src, index or dst", fn);
  if (n < 1 || n_src < 1 || H < 1 || W < 1 || h < 1 || w < 1) return set_err(nullptr, EDV_ERR_ARG, "%s: empty problem", fn);
  if (stride_n < 1 || stride_y < 1 || stride_x < 1 || stride_c < 1)
    return set_err(nullptr, EDV_ERR_ARG, "%s: strides must be positive", fn);
  // the last byte of the source must have a 64-bit offset (the kernel forms it as n*sn + y*sy + x*sx + c*sc)
  const __int128 extent = (__int128)(n_src - 1) * stride_n + (__int128)(H - 1) * stride_y + (__int128)(W - 1) * stride_x +
                          (__int128)2 * stride_c;
  if (extent > (__int128)INT64_MAX) return set_err(nullptr, EDV_ERR_ARG, "%s: source extent overflows 64-bit offsets", fn);
  for (int i = 0; i < n; ++i)
    if (index_host[i] < 0 || index_host[i] >= n_src)
      return set_err(nullptr, EDV_ERR_ARG, "%s: index[%d] = %lld outside [0, %d)", fn, i, (long long)index_host[i], n_src);
  Launch L;
  L.stream = (cudaStream_t)stream;
  cubic_resize_u8(L, src, H, W, stride_n, stride_y, stride_x, stride_c, index_host, n, dst, h, w);
  return finish(L);
}

int edv_op_layernorm(int dtype, const float* X, const float* gamma, const float* beta, void* Y, int M, int D, float eps, int grp,
                     int skip, const float* add, int add_div, int add_mod, void* stream) {
  if (dtype < EDV_F32 || dtype > EDV_F16) return set_err(nullptr, EDV_ERR_ARG, "edv_op_layernorm: bad dtype %d", dtype);
  if (!X || !gamma || !beta || !Y) return set_err(nullptr, EDV_ERR_ARG, "edv_op_layernorm: null argument");
  if (M < 1) return set_err(nullptr, EDV_ERR_ARG, "edv_op_layernorm: empty problem");
  if (grp < 0 || (grp == 0 && skip != 0) || (grp > 0 && (skip >= grp || -skip > grp)))
    return set_err(nullptr, EDV_ERR_ARG, "edv_op_layernorm: skip %d outside (-grp, grp) for grp %d", skip, grp);
  if (add && (add_div < 1 || add_mod < 1)) return set_err(nullptr, EDV_ERR_ARG, "edv_op_layernorm: add_div and add_mod must be >= 1");
  if (!aligned16(X) || !aligned16(gamma) || !aligned16(beta) || !aligned16(add))
    return set_err(nullptr, EDV_ERR_ARG, "edv_op_layernorm: X, gamma, beta and add must be 16-byte aligned");
  Launch L;
  L.stream = (cudaStream_t)stream;
  layernorm(L, dtype, X, gamma, beta, Y, M, D, eps, grp, skip, add, add ? add_div : 1, add ? add_mod : 1);
  return finish(L);
}

int edv_op_preprocess_patches(int dtype, const void* src, int u8, void* out, int F, int H, int W, int h, int w, int normalize,
                              void* stream) {
  if (dtype < EDV_F32 || dtype > EDV_F16) return set_err(nullptr, EDV_ERR_ARG, "edv_op_preprocess_patches: bad dtype %d", dtype);
  if (!src || !out) return set_err(nullptr, EDV_ERR_ARG, "edv_op_preprocess_patches: null src or out");
  if (F < 1 || H < 1 || W < 1 || h < 14 || w < 14 || h % 14 || w % 14)
    return set_err(nullptr, EDV_ERR_ARG, "edv_op_preprocess_patches: frames must be non-empty and h, w multiples of 14");
  if (u8 && (H != h || W != w)) return set_err(nullptr, EDV_ERR_ARG, "edv_op_preprocess_patches: uint8 frames must be at network resolution");
  if (!aligned16(out)) return set_err(nullptr, EDV_ERR_ARG, "edv_op_preprocess_patches: out must be 16-byte aligned");
  Launch L;
  L.stream = (cudaStream_t)stream;
  preprocess_patches(L, dtype, src, u8 != 0, out, F, H, W, h, w, KPATCH, normalize ? 1 : 0);
  return finish(L);
}

int edv_op_tokens_to_patches(int dtype, const float* x, void* out, long long Mp, int P, int D, int cls, void* stream) {
  if (dtype < EDV_F32 || dtype > EDV_F16) return set_err(nullptr, EDV_ERR_ARG, "edv_op_tokens_to_patches: bad dtype %d", dtype);
  if (!x || !out) return set_err(nullptr, EDV_ERR_ARG, "edv_op_tokens_to_patches: null x or out");
  if (Mp < 1 || P < 1 || Mp % P || D < 4 || D % 4 || (cls != 0 && cls != 1))
    return set_err(nullptr, EDV_ERR_ARG, "edv_op_tokens_to_patches: needs Mp a multiple of P, D %% 4 == 0, cls 0 or 1");
  if (!aligned16(x) || !aligned16(out)) return set_err(nullptr, EDV_ERR_ARG, "edv_op_tokens_to_patches: x and out must be 16-byte aligned");
  Launch L;
  L.stream = (cudaStream_t)stream;
  tokens_to_patches(L, dtype, x, out, Mp, P, D, cls);
  return finish(L);
}

int edv_op_rowln_act(int dtype, const void* x, const float* gamma, const float* beta, void* y, long long M, int C, int Cr, float eps,
                     int gelu, void* stream) {
  if (dtype < EDV_F32 || dtype > EDV_F16) return set_err(nullptr, EDV_ERR_ARG, "edv_op_rowln_act: bad dtype %d", dtype);
  if (!x || !gamma || !beta || !y) return set_err(nullptr, EDV_ERR_ARG, "edv_op_rowln_act: null argument");
  if (M < 1 || Cr < 1 || Cr > C) return set_err(nullptr, EDV_ERR_ARG, "edv_op_rowln_act: needs M >= 1 and 1 <= Cr <= C");
  Launch L;
  L.stream = (cudaStream_t)stream;
  rowln_act(L, dtype, x, gamma, beta, y, M, C, Cr, eps, gelu ? 1 : 0);
  return finish(L);
}

int edv_op_resblock_add(int dtype, float* x, const void* r, const float* gamma, const float* beta, long long Mp, int P, int D, float eps,
                        int cls, void* stream) {
  if (dtype < EDV_F32 || dtype > EDV_F16) return set_err(nullptr, EDV_ERR_ARG, "edv_op_resblock_add: bad dtype %d", dtype);
  if (!x || !r || !gamma || !beta) return set_err(nullptr, EDV_ERR_ARG, "edv_op_resblock_add: null argument");
  if (Mp < 1 || P < 1 || Mp % P || D < 1 || (cls != 0 && cls != 1))
    return set_err(nullptr, EDV_ERR_ARG, "edv_op_resblock_add: needs Mp a multiple of P, D >= 1, cls 0 or 1");
  Launch L;
  L.stream = (cudaStream_t)stream;
  resblock_add(L, dtype, x, r, gamma, beta, Mp, P, D, eps, cls);
  return finish(L);
}

int edv_op_im2col3x3(int dtype, const void* x, void* out, int F, int H, int W, int C, int stride, void* stream) {
  if (dtype < EDV_F32 || dtype > EDV_F16) return set_err(nullptr, EDV_ERR_ARG, "edv_op_im2col3x3: bad dtype %d", dtype);
  if (!x || !out) return set_err(nullptr, EDV_ERR_ARG, "edv_op_im2col3x3: null x or out");
  if (F < 1 || H < 1 || W < 1 || C < 8 || C % 8 || stride < 1 || stride > 2)
    return set_err(nullptr, EDV_ERR_ARG, "edv_op_im2col3x3: needs a non-empty map, C %% 8 == 0 and stride 1 or 2");
  if (!aligned16(x) || !aligned16(out)) return set_err(nullptr, EDV_ERR_ARG, "edv_op_im2col3x3: x and out must be 16-byte aligned");
  Launch L;
  L.stream = (cudaStream_t)stream;
  im2col3x3(L, dtype, x, out, F, H, W, C, (H - 1) / stride + 1, (W - 1) / stride + 1, stride);
  return finish(L);
}

int edv_op_geglu_pair(int dtype, const void* hg, void* out, long long M, int C4, void* stream) {
  if (dtype < EDV_F32 || dtype > EDV_F16) return set_err(nullptr, EDV_ERR_ARG, "edv_op_geglu_pair: bad dtype %d", dtype);
  if (!hg || !out) return set_err(nullptr, EDV_ERR_ARG, "edv_op_geglu_pair: null hg or out");
  if (M < 1 || C4 < 64 || C4 % 64) return set_err(nullptr, EDV_ERR_ARG, "edv_op_geglu_pair: needs M >= 1 and C4 a multiple of 64");
  Launch L;
  L.stream = (cudaStream_t)stream;
  geglu_pair(L, dtype, hg, out, M, C4);
  return finish(L);
}

int edv_op_head_dot(int dtype, const void* x, const float* w, float* out, long long M, int C, float sig_sign, void* stream) {
  if (dtype < EDV_F32 || dtype > EDV_F16) return set_err(nullptr, EDV_ERR_ARG, "edv_op_head_dot: bad dtype %d", dtype);
  if (!x || !w || !out) return set_err(nullptr, EDV_ERR_ARG, "edv_op_head_dot: null x, w or out");
  if (M < 1 || C < 8 || C % 8) return set_err(nullptr, EDV_ERR_ARG, "edv_op_head_dot: needs M >= 1 and C a multiple of 8");
  if (!aligned16(x)) return set_err(nullptr, EDV_ERR_ARG, "edv_op_head_dot: x must be 16-byte aligned");
  Launch L;
  L.stream = (cudaStream_t)stream;
  head_dot(L, dtype, x, w, out, M, C, sig_sign);
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
