// (a8) GETAM from row-0 quantities and (a9) affinity refinement.
// Reference: DPT/ACR.py:177-215 (getam), infer_cam.py:164-165 (patch_aff = sum over blocks of the
// patch x patch part of the head-mean map) and infer_cam.py:184 (matmul(patch_aff, cam)).
#include "common.cuh"

namespace {

// max(v, 0) that keeps a NaN, as torch's clamp(min=0) and relu do (fmaxf would return 0).
__device__ __forceinline__ float relu_nan(float v) { return v < 0.f ? 0.f : v; }

// One thread per token j, blockIdx.y = sample.  p/g: [L,S,H,N] (S = 1 for the single-image entry).  See acr_b200.h for `func`.
__global__ void __launch_bounds__(256)
getam_row0_kernel(const float* __restrict__ p, const float* __restrict__ g, int S, int L, int H, int N,
                  int start_layer, int func, int skip, float* __restrict__ cam_out, float* __restrict__ cam_rows) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  const int s = blockIdx.y;
  if (j >= N) return;
  cam_out += (long long)s * (N - skip);
  if (cam_rows) cam_rows += (long long)s * L * N;
  const float invH = 1.f / (float)H;
  float total = 0.f;
  for (int l = 0; l < L; ++l) {
    float pos_g = 0.f, pos_gp = 0.f;
    for (int h = 0; h < H; ++h) {
      const long long o = (((long long)l * S + s) * H + h) * N + j;
      const float gv = g[o];
      pos_g += relu_nan(gv);
      if (func >= 2) pos_gp += relu_nan(gv * p[o]);
    }
    pos_g *= invH;
    pos_gp *= invH;
    float c;
    switch (func) {
      case 0: c = pos_g; break;
      case 1: c = pos_g * pos_g; break;
      case 2: c = pos_gp; break;
      default: c = pos_gp * pos_g; break;
    }
    if (cam_rows) cam_rows[(long long)l * N + j] = c;
    if (l >= start_layer) total += c;
  }
  if (j >= skip) cam_out[j - skip] = relu_nan(total);
}

// A[b,i,:] = sum_l attn[b,l,i+1,1:] (optionally divided by its row sum).  One CTA per (b,i).
__global__ void __launch_bounds__(256)
affinity_sum_kernel(const float* __restrict__ attn, int L, int N, int normalize, float* __restrict__ A) {
  __shared__ float red[32];
  const int Np = N - 1;
  const int i = blockIdx.x, b = blockIdx.y;
  const float* src = attn + ((long long)b * L * N + (i + 1)) * (long long)N + 1;
  float* dst = A + ((long long)b * Np + i) * (long long)Np;
  float rs = 0.f;
  for (int j = threadIdx.x; j < Np; j += blockDim.x) {
    float s = 0.f;
    for (int l = 0; l < L; ++l) s += __ldg(src + (long long)l * N * N + j);
    dst[j] = s;
    rs += s;
  }
  if (normalize) {
    rs = acr::block_sum(rs, red);
    const float inv = 1.f / rs;
    for (int j = threadIdx.x; j < Np; j += blockDim.x) dst[j] *= inv;
  }
}

}  // namespace

extern "C" int acr_getam_row0(const float* p_row0, const float* g_row0, int L, int H, int N,
                              int start_layer, int func, int skip,
                              float* cam_out, float* cam_rows, void* stream) {
  ACR_REQUIRE(p_row0 && g_row0 && cam_out, ACR_E_INVAL, "acr_getam_row0: null pointer");
  ACR_REQUIRE(L > 0 && H > 0 && N > 1, ACR_E_INVAL, "acr_getam_row0: bad shape");
  ACR_REQUIRE(start_layer >= 0 && start_layer < L, ACR_E_INVAL, "acr_getam_row0: start_layer %d outside [0,%d)", start_layer, L);
  ACR_REQUIRE(func >= 0 && func <= 3, ACR_E_INVAL, "acr_getam_row0: unknown func %d", func);
  ACR_REQUIRE(skip >= 1 && skip < N, ACR_E_INVAL, "acr_getam_row0: bad skip");
  getam_row0_kernel<<<(N + 255) / 256, 256, 0, (cudaStream_t)stream>>>(p_row0, g_row0, 1, L, H, N, start_layer, func, skip, cam_out, cam_rows);
  return acr::check_launch("getam_row0_kernel");
}

extern "C" int acr_getam_row0_batch(const float* p_row0, const float* g_row0, int S, int L, int H, int N,
                                    int start_layer, int func, int skip, float* cam_out, void* stream) {
  ACR_REQUIRE(p_row0 && g_row0 && cam_out, ACR_E_INVAL, "acr_getam_row0_batch: null pointer");
  ACR_REQUIRE(S > 0 && S <= 65535 && L > 0 && H > 0 && N > 1, ACR_E_INVAL, "acr_getam_row0_batch: bad shape");
  ACR_REQUIRE(start_layer >= 0 && start_layer < L, ACR_E_INVAL, "acr_getam_row0_batch: start_layer %d outside [0,%d)", start_layer, L);
  ACR_REQUIRE(func >= 0 && func <= 3, ACR_E_INVAL, "acr_getam_row0_batch: unknown func %d", func);
  ACR_REQUIRE(skip >= 1 && skip < N, ACR_E_INVAL, "acr_getam_row0_batch: bad skip");
  getam_row0_kernel<<<dim3((N + 255) / 256, S), 256, 0, (cudaStream_t)stream>>>(p_row0, g_row0, S, L, H, N, start_layer, func, skip, cam_out, nullptr);
  return acr::check_launch("getam_row0_kernel");
}

extern "C" int acr_affinity_sum(const float* attn, int B, int L, int N, int normalize, float* A, void* stream) {
  ACR_REQUIRE(attn && A, ACR_E_INVAL, "acr_affinity_sum: null pointer");
  ACR_REQUIRE(B > 0 && B <= 65535 && L > 0 && N > 1, ACR_E_INVAL, "acr_affinity_sum: bad shape");
  dim3 grid(N - 1, B);
  affinity_sum_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(attn, L, N, normalize, A);
  return acr::check_launch("affinity_sum_kernel");
}

extern "C" int acr_affinity_refine(const float* A, const float* cam, int B, int Np, int C, int t,
                                   float* out, float* tmp, void* stream) {
  ACR_REQUIRE(A && cam && out, ACR_E_INVAL, "acr_affinity_refine: null pointer");
  ACR_REQUIRE(B > 0 && B <= 65535 && Np > 0 && C > 0 && t >= 1, ACR_E_INVAL, "acr_affinity_refine: bad shape");
  ACR_REQUIRE(t == 1 || tmp, ACR_E_INVAL, "acr_affinity_refine: tmp required when t>1");
  const acr::Mat la{(long long)Np * Np, 0, Np, 1};
  const acr::Mat lc{(long long)Np * C, 0, C, 1};
  // Ping-pong so that the t-th product lands in `out`.
  const float* src = cam;
  for (int s = 0; s < t; ++s) {
    float* dst = ((t - 1 - s) % 2 == 0) ? out : tmp;
    if (int e = acr::launch_sgemm(A, la, src, lc, dst, lc, Np, C, Np, B, 1, 1.f, (cudaStream_t)stream)) return e;
    src = dst;
  }
  return 0;
}
