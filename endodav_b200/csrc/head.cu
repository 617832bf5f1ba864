// Launcher of the fused disparity-head tail (head_fused.cuh).
#include "ops.h"
#include "head_fused.cuh"

namespace edv {

// fused upsample -> conv3x3 (Cin -> 32) -> ReLU -> 1x1 -> ReLU|sigmoid  (head_fused.cuh)
template <typename T, int CIN>
void launch_head_fused(Launch& L, const void* x, const void* w, const float* bias, const float* head_w, float* out, int F,
                       int H1, int W1, int OH, int OW, float sig_sign) {
  using namespace tc;
  constexpr auto kern = head_fused_kernel<T, CIN>;
  smem_opt_in<kern>((int)hf_smem_bytes<CIN>());
  const int tiles_x = (OW + HF_TW - 1) / HF_TW, tiles_y = (OH + HF_TH - 1) / HF_TH;
  const long long total = (long long)F * tiles_x * tiles_y;
  if (total > 0x7fffffffLL) return L.fail(EDV_ERR_ARG, "head_fused: too many tiles");
  const int grid = (int)std::min<long long>(total, num_sms());
  // algorithmic bytes: the low-resolution map once + one float per output pixel (SURVEY.md 8(d))
  L.note(2.0 * F * OH * OW * 32.0 * (9 * CIN + 1), (double)F * H1 * W1 * CIN * sizeof(T) + (double)F * OH * OW * 4);
  edv::launch_k(kern, dim3(grid), dim3(HF_THREADS), hf_smem_bytes<CIN>(), L.stream, (const T*)x, (const T*)w, bias, head_w, out, F, H1, W1, OH, OW,
                                                           sig_sign, tiles_x, tiles_y, (int)total);
  L.check("head_fused");
}

bool head_fused_supported(int dtype, int Cin) { return dtype != EDV_F32 && (Cin == 32 || Cin == 128); }

void head_fused(Launch& L, int dtype, const void* x, const void* w, const float* bias, const float* head_w,
                       float* out, int F, int H1, int W1, int OH, int OW, int Cin, float sig_sign) {
  if (!L.ok()) return;
  if (!head_fused_supported(dtype, Cin)) return L.fail(EDV_ERR_ARG, "head_fused: 16-bit dtype and Cin in {32,128} only");
#define EDV_HF_CASE(T_, C_) launch_head_fused<T_, C_>(L, x, w, bias, head_w, out, F, H1, W1, OH, OW, sig_sign)
  if (dtype == EDV_BF16) { if (Cin == 32) EDV_HF_CASE(bf16, 32); else EDV_HF_CASE(bf16, 128); }
  else { if (Cin == 32) EDV_HF_CASE(f16, 32); else EDV_HF_CASE(f16, 128); }
#undef EDV_HF_CASE
}

}  // namespace edv
