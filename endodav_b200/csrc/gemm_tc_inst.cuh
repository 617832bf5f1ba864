// Host launchers of the tcgen05 GEMM family (gemm_tc.cuh, gemm_bres.cuh, gemm_ln.cuh, conv_halo.cuh).  Included by
// the gemm_tc_*.cu translation units, each of which explicitly instantiates one (dtype, lin|conv) slice.
#pragma once
#include "ops.h"
#include "gemm_tc.cuh"
#include "gemm_bres.cuh"
#include "gemm_ln.cuh"
#include "conv_halo.cuh"

namespace edv {

// the TMA-store epilogue handles 16-bit row-major outputs of the EDV_EPI_TMA_KINDS only
inline bool gemm_tma_out_ok(const GemmArgs& a) {
  using namespace tc;
  if (a.conv) return false;
  switch (a.e.kind) {
#define EDV_KIND_LABEL(F_) case F_:
    EDV_EPI_TMA_KINDS(EDV_KIND_LABEL) break;
#undef EDV_KIND_LABEL
    default: return false;
  }
  if (a.e.map != MAP_LINEAR || a.e.out_f32 || !a.e.out) return false;
  if ((a.e.ldo * 2) % 16 != 0 || ((uintptr_t)a.e.out & 15) != 0) return false;
  return true;
}

template <typename T, int BN, int BK, bool CONV>
void launch_gemm_tc_inst(Launch& L, int dtype, const GemmArgs& a) {
  using namespace tc;
  CUtensorMap tmA, tmB;
  ConvTile ct{};
  long long m_tiles;
  const int swz = BK * 2;
  if (CONV) {
    ct.H = a.H; ct.W = a.Wd; ct.C = a.C;
    pick_conv_tile(a.H, a.Wd, &ct.th, &ct.tw);
    ct.tiles_y = (a.H + ct.th - 1) / ct.th;
    ct.tiles_x = (a.Wd + ct.tw - 1) / ct.tw;
    m_tiles = (long long)a.F * ct.tiles_y * ct.tiles_x;
    uint64_t dims[4] = {(uint64_t)a.C, (uint64_t)a.Wd, (uint64_t)a.H, (uint64_t)a.F};
    uint64_t str[3] = {(uint64_t)a.C * 2, (uint64_t)a.C * a.Wd * 2, (uint64_t)a.C * a.Wd * a.H * 2};
    uint32_t box[4] = {(uint32_t)BK, (uint32_t)ct.tw, (uint32_t)ct.th, 1};
    if (!make_tmap(L, &tmA, dtype, a.A, 4, dims, str, box, swz)) return;
  } else {
    m_tiles = (a.M + GT_BM - 1) / GT_BM;
    if (!make_tmap_2d(L, &tmA, dtype, a.A, a.K, a.M, a.lda * 2, BK, GT_BM, swz)) return;
  }
  if (!make_tmap_2d(L, &tmB, dtype, a.W, a.K, a.N, a.K * 2, BK, BN, swz)) return;
  // TMA-store epilogue: output tensor map over C [M rows, N cols] (row pitch ldo), box 16 columns x 128 rows, 32B swizzle
  CUtensorMap tmC;
  memset(&tmC, 0, sizeof tmC);
  GemmArgs a2 = a;
  if (!CONV && BN % 64 == 0 && gemm_tma_out_ok(a)) {
    if (!make_tmap_2d(L, &tmC, dtype, a.e.out, a.N, a.M, a.e.ldo * 2, 16, GT_BM, 32)) return;
    a2.e.kind |= tc::EF_TMA_OUT;
  }
  const int kblocks = a.K / BK;
  const int stage_bytes = gt_stage_bytes<BN, BK>();
  const size_t stg_bytes = 16 * (size_t)GT_STG_WORDS * 4 + 16 * 128 * 4;   // + per-warp bias slices   // epilogue transposition buffers
  int stages = (int)((220 * 1024 - stg_bytes - 2048) / stage_bytes);  // one persistent CTA per SM owns the shared memory
  if (stages > 8) stages = 8;
  if (stages < 2) stages = 2;
  const size_t smem = (size_t)stages * stage_bytes + 1024 /*align*/ + (2 * stages + 4) * 8 + 16 + stg_bytes;
  constexpr auto kern = gemm_tc_kernel<T, BN, BK, CONV>;
  smem_opt_in<kern>(226 * 1024);
  const int n_tiles = a.N / BN;
  const long long total = m_tiles * n_tiles;
  if (total > 0x7fffffffLL) return L.fail(EDV_ERR_ARG, "gemm_tc: too many tiles");
  const int grid = (int)std::min<long long>(total, num_sms());
  (void)kblocks;
  note_gemm(L, a, 2);
  L.kernel = std::string(CONV ? "gemm_tc_conv<" : "gemm_tc<") + "BN=" + std::to_string(BN) + ",BK=" + std::to_string(BK) + ",kind=" +
             kind_label(a.e.kind) + (CONV ? ">" : (a2.e.kind != a.e.kind ? ",tma=1>" : ",tma=0>"));
  edv::launch_k(kern, dim3(grid), dim3(GT_THREADS), smem, L.stream, tmA, tmB, tmC, a2.e, a.M, a.N, a.K, stages, ct, n_tiles, (int)total);
  L.check("gemm_tc");
}

// 64-channel 3x3 convs with halo reuse (conv_halo.cuh)
template <typename T, int BN> void launch_conv_halo(Launch& L, const GemmArgs& a) {
  using namespace tc;
  constexpr auto kern = conv3x3_halo_kernel<T, 64, BN>;
  smem_opt_in<kern>((int)ch_smem_bytes<64, BN>());
  const int tiles_x = (a.Wd + CH_TW - 1) / CH_TW, tiles_y = (a.H + CH_TH - 1) / CH_TH;
  const long long total = (long long)a.F * tiles_x * tiles_y;
  if (total > 0x7fffffffLL) return L.fail(EDV_ERR_ARG, "conv_halo: too many tiles");
  const int grid = (int)std::min<long long>(total, num_sms());
  note_gemm(L, a, 2);
  L.kernel = "conv_halo<BN=" + std::to_string(BN) + ",kind=" + kind_label(a.e.kind) + ">";
  edv::launch_k(kern, dim3(grid), dim3(CH_THREADS), ch_smem_bytes<64, BN>(), L.stream, (const T*)a.A, (const T*)a.W, a.e, a.F, a.H, a.Wd, tiles_x,
                                                               tiles_y, (int)total);
  L.check("conv_halo");
}

inline bool conv_halo_ok(const GemmArgs& a) {
  return a.conv && a.stride == 1 && a.C == 64 && (a.N == 64 || a.N == 32) &&
         (a.e.act == ACT_NONE || a.e.act == ACT_RELU || a.e.act == ACT_SIGMOID) && a.e.map == MAP_LINEAR;
}

inline int gemm_tc_pick_bk(const GemmArgs& a) { return (a.conv ? (a.C % 64 != 0) : (a.K % 64 != 0)) ? 32 : 64; }

inline int gemm_tc_pick_bn(const GemmArgs& a, int bk) {
  int bn;
  if (a.e.act == ACT_GEGLU) bn = 128;
  else if (a.e.act == ACT_HEAD) bn = 32;
  else if (bk == 64 && a.N % 256 == 0) bn = 256;   // wide tiles halve the shared-memory traffic per FLOP
  else if (bk == 64 && a.N % 192 == 0) bn = 192;
  else bn = (a.N % 128 == 0) ? 128 : (a.N % 64 == 0) ? 64 : 32;
  if (a.e.map == MAP_PIXSHUF && (a.e.ps_c % bn != 0 && bn % a.e.ps_c != 0)) bn = 64;
  return bn;
}

template <typename T, bool CONV> void launch_gemm_tc_any(Launch& L, int dtype, const GemmArgs& a) {
  const int bk = gemm_tc_pick_bk(a);
  if ((a.conv ? a.C : a.K) % bk != 0) return L.fail(EDV_ERR_ARG, "gemm_tc: K (or conv C) must be a multiple of 32");
  if (a.conv && a.stride != 1) return L.fail(EDV_ERR_ARG, "gemm_tc: conv stride must be 1");
  const int bn = gemm_tc_pick_bn(a, bk);
  if (a.N % bn != 0) return L.fail(EDV_ERR_ARG, "gemm_tc: N must be a multiple of 32");
  if (a.e.act == ACT_HEAD && a.N != 32) return L.fail(EDV_ERR_ARG, "gemm_tc: head epilogue needs N == 32");
#define EDV_TC_CASE(BN_, BK_) \
  if (bn == BN_ && bk == BK_) return launch_gemm_tc_inst<T, BN_, BK_, CONV>(L, dtype, a);
  EDV_TC_CASE(256, 64)
  EDV_TC_CASE(192, 64)
  EDV_TC_CASE(128, 64)
  EDV_TC_CASE(64, 64)
  EDV_TC_CASE(32, 64)
  EDV_TC_CASE(128, 32)
  EDV_TC_CASE(64, 32)
  EDV_TC_CASE(32, 32)
#undef EDV_TC_CASE
  L.fail(EDV_ERR_ARG, "gemm_tc: no instantiation");
}

#ifdef EDV_GEMM_TU_LIN
// B-resident GEMM (gemm_bres.cuh): short K, 16-bit output through the TMA-store epilogue
constexpr size_t GB_SMEM_MAX = 232448 - 1024;   // 227 KB opt-in limit minus the alignment slack

template <typename T, int BN> bool launch_gemm_bres(Launch& L, int dtype, const GemmArgs& a) {
  using namespace tc;
  const int kblocks = a.K / 64;
  const size_t b_bytes = (size_t)kblocks * BN * 128;
  const size_t fixed = b_bytes + 4 * GT_OUT_SUB_BYTES + 4 * 64 * 4 + 512;
  if (fixed + 2 * GB_A_STAGE > GB_SMEM_MAX) return false;
  int stages = (int)((GB_SMEM_MAX - fixed) / GB_A_STAGE);
  if (stages > 8) stages = 8;
  CUtensorMap tmA, tmB, tmC;
  if (!make_tmap_2d(L, &tmA, dtype, a.A, a.K, a.M, a.lda * 2, 64, GT_BM, 128)) return true;
  if (!make_tmap_2d(L, &tmB, dtype, a.W, a.K, a.N, a.K * 2, 64, BN, 128)) return true;
  if (!make_tmap_2d(L, &tmC, dtype, a.e.out, a.N, a.M, a.e.ldo * 2, 16, GT_BM, 32)) return true;
  constexpr auto kern = gemm_bres_kernel<T, BN>;
  smem_opt_in<kern>(232448);
  const int n_tiles = a.N / BN;
  const int m_tiles = (a.M + GT_BM - 1) / GT_BM;
  int grid = num_sms();
  if (grid < n_tiles) return false;
  if ((long long)m_tiles * n_tiles < grid) grid = std::max(n_tiles, m_tiles * n_tiles);
  const size_t smem = fixed + (size_t)stages * GB_A_STAGE + 1024;
  GemmArgs a2 = a;
  a2.e.kind |= EF_TMA_OUT;
  note_gemm(L, a, 2);
  L.kernel = "gemm_bres<BN=" + std::to_string(BN) + ">";
  edv::launch_k(kern, dim3(grid), dim3(GB_THREADS), smem, L.stream, tmA, tmB, tmC, a2.e, a.M, a.K, stages, n_tiles, m_tiles);
  L.check("gemm_bres");
  return true;
}

template <typename T>
void launch_gemm_ln(Launch& L, int dtype, const void* A, const void* W, const float* bias, float* x, void* xn, const float* gamma,
                    const float* beta, float eps, int M, int K, int do_ln, long long* tim) {
  using namespace tc;
  CUtensorMap tmA, tmB, tmX, tmXn;
  if (!make_tmap_2d(L, &tmA, dtype, A, K, M, K * 2, 64, GT_BM, 128)) return;
  if (!make_tmap_2d(L, &tmB, dtype, W, K, GL_N, K * 2, 64, GL_HN, 128)) return;
  if (!make_tmap_2d(L, &tmX, EDV_F32, x, GL_N, M, GL_N * 4, 16, GT_BM, 64)) return;
  if (!make_tmap_2d(L, &tmXn, dtype, do_ln ? xn : (const void*)x, GL_N, M, GL_N * 2, 16, GT_BM, 32)) return;
  constexpr auto kern = gemm_ln_kernel<T>;
  smem_opt_in<kern>((int)GL_SMEM);
  const int m_tiles = (M + GT_BM - 1) / GT_BM;
  const int grid = 2 * std::min(m_tiles, num_sms() / 2);   // clusters of two CTAs, one 128-row tile per pair at a time
  // algorithmic work: 2 M N K; bytes: A + W + the fp32 stream read and written once + xn written once
  L.note(2.0 * M * GL_N * K, ((double)M * K + (double)GL_N * K) * 2 + (double)M * GL_N * (8 + (do_ln ? 2 : 0)));
  edv::launch_k(kern, dim3(grid), dim3(GL_THREADS), GL_SMEM, L.stream, tmA, tmB, tmX, tmXn, bias, gamma, beta, eps, M, K, m_tiles, do_ln, tim);
  L.check("gemm_ln");
}

#ifdef EDV_GEMM_TU_LN
bool gemm_ln_supported(int dtype, int N, int K) {
  return dtype != EDV_F32 && N == tc::GL_N && K % 64 == 0 && K >= 64;
}
void gemm_ln(Launch& L, int dtype, const void* A, const void* W, const float* bias, float* x, void* xn, const float* gamma,
             const float* beta, float eps, int M, int N, int K, int do_ln, long long* tim) {
  if (!L.ok()) return;
  if (!gemm_ln_supported(dtype, N, K)) return L.fail(EDV_ERR_ARG, "gemm_ln: needs a 16-bit dtype, N == 384 and K % 64 == 0");
  if (dtype == EDV_BF16) launch_gemm_ln<bf16>(L, dtype, A, W, bias, x, xn, gamma, beta, eps, M, K, do_ln, tim);
  else launch_gemm_ln<f16>(L, dtype, A, W, bias, x, xn, gamma, beta, eps, M, K, do_ln, tim);
}
#endif

// linear GEMMs (2-D A operand)
template <typename T> void launch_gemm_tc_lin(Launch& L, int dtype, const GemmArgs& a) {
  if (gemm_tma_out_ok(a) && a.K % 64 == 0 && a.K <= 384 && a.lda == a.K && a.M >= 2048) {
    if (a.N % 192 == 0) { if (launch_gemm_bres<T, 192>(L, dtype, a)) return; }
    else if (a.N % 128 == 0) { if (launch_gemm_bres<T, 128>(L, dtype, a)) return; }
    else if (a.N % 64 == 0) { if (launch_gemm_bres<T, 64>(L, dtype, a)) return; }
  }
  launch_gemm_tc_any<T, false>(L, dtype, a);
}
#endif

#ifdef EDV_GEMM_TU_CONV
// 3x3 convolutions: halo-reuse kernel for the 64-channel maps, TMA implicit GEMM otherwise
template <typename T> void launch_gemm_tc_conv(Launch& L, int dtype, const GemmArgs& a) {
  if (conv_halo_ok(a)) {
    if (a.N == 64) launch_conv_halo<T, 64>(L, a);
    else launch_conv_halo<T, 32>(L, a);
    return;
  }
  launch_gemm_tc_any<T, true>(L, dtype, a);
}
#endif

}  // namespace edv
