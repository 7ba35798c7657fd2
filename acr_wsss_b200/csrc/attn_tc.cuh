// Shared pieces of the fused tcgen05 attention kernels (attn_tc.cu: forward / head mean / delta pass, attn_bwd_tc.cu: backward).
#pragma once
#include "common.cuh"
#include "tc_common.cuh"

namespace acr_attn {

constexpr int BM = 128;               // query rows per tile
constexpr int BN = 128;               // key rows per tile
constexpr int HD = 64;                // head dim (128-byte bf16 rows = one SWIZZLE_128B atom row)
constexpr uint32_t TILE_BYTES = BM * HD * 2;
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;
constexpr int MEAN_MAX_H = 32;
// dQ is summed over the key tiles in 64-bit fixed point (value * 2^40, resolution 2^-40): integer addition is associative, so
// the order in which the key tiles' TMA reduce-adds land does not change a bit of the result.  Range: the host passes the
// largest per-tile magnitude that kt partials can sum without leaving int64 (dq_fix_limit: 2^(62 - ceil(log2 kt)) in fixed
// units, i.e. |partial| < 2^19 for N <= 1024); a partial beyond it, or not finite, is not added but marks its query row, and
// bwd_dq_convert_kernel writes that row of dQ as NaN (a NaN or overflow propagates, as it would through an fp32 sum).
constexpr float kDqFix = 1099511627776.0f;            // 2^40
constexpr float kDqUnfix = 1.0f / 1099511627776.0f;   // 2^-40
inline float dq_fix_limit(int kt) {
  int lg = 0;
  while ((1 << lg) < kt) ++lg;
  return ldexpf(1.0f, 62 - lg);
}

constexpr uint32_t IDESC_S = tc::idesc_bf16_f32(128, 128, 0, 0);   // S = Q K^T : A, B K-major
constexpr uint32_t IDESC_PV = tc::idesc_bf16_f32(128, 64, 0, 1);   // O = P V   : A K-major, B = V MN-major
constexpr uint32_t IDESC_DQ = tc::idesc_bf16_f32(128, 64, 1, 1);   // dV = P^T dO, dK = dS^T Q : A MN-major (smem), B MN-major

// Sign-code form of G (acr_consistency_fwd_bwd): one byte per element = top byte of +-0.5f; strides in bytes.
struct GCode {
  const unsigned char* ptr;
  long long bs, ld;
  float w_cls, w_aff;
  const float* scale;     // optional device scalar
};
__device__ __forceinline__ float gcode_weight(const GCode& gc, int q, float invH) {   // 2*w*scale/H of query row q
  const float sc = gc.scale ? __ldg(gc.scale) : 1.f;
  return 2.f * invH * sc * (q == 0 ? gc.w_cls : gc.w_aff);
}
// byte k (0..3) of a word moved to the top byte of an fp32: 0x3F -> +0.5f, 0xBF -> -0.5f, 0x00 -> 0
#define ACR_CODE_F(word, k) __uint_as_float(__byte_perm((word), 0u, 0x0444u | ((k) << 12)))

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn get_encode_fn();
// bf16 tensor [B, N, S*H, D] (S = 3 for qkv, 1 for out / d_out) viewed as 4-D (d, sh, n, b); box = 128 rows x 64 d.
int make_tmap(CUtensorMap* m, const void* base, int B, int N, int SH, int D);

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-device attribute: set it once per (kernel, device).
template <typename K>
int set_max_smem(K kernel, size_t bytes, bool* done /* [64] */) {
  int dev = 0;
  ACR_CUDA(cudaGetDevice(&dev));
  if (dev >= 0 && dev < 64 && done[dev]) return 0;
  ACR_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  if (dev >= 0 && dev < 64) done[dev] = true;
  return 0;
}

// backward kernel launcher (attn_bwd_tc.cu)
int launch_attn_bwd(const CUtensorMap& tmap_qkv, const CUtensorMap& tmap_do, const CUtensorMap& tmap_dq, const float* lse, const float* delta,
                    const float* g_mean, long long g_bs, long long g_ld, const GCode& gc, __nv_bfloat16* d_qkv, float* g_row0,
                    int* dq_bad, int B, int N, int H, float scale, cudaStream_t st);

}  // namespace acr_attn
