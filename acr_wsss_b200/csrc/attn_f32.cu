// (a1/a2) Exact fp32 attention path that materialises P = softmax(QK^T * scale) [B,H,N,N] and, in the
// backward, dP -- i.e. the data flow of the reference (models/vision_transformer.py:198-214 and the
// save_attn / save_attn_gradients hook protocol :186-196), written as plain CUDA-core kernels.
// It exists for (i) 1e-3 fp32 parity checks, (ii) the get_attn()/get_attn_gradients() accessors and
// (iii) an on-device cross-check of the fused tcgen05 path.  It is NOT the fast path.
//
// One strided, batched SGEMM kernel serves all six contractions (QK^T, PV, dO V^T, P^T dO, dS K, dS^T Q);
// row softmax, head mean and the softmax backward (with the dense affinity-gradient term) are separate
// streaming kernels.
#include "common.cuh"

using acr::Mat;

namespace {

constexpr int TM = 64, TN = 64, TK = 16;

// C[m,n] = alpha * sum_k A[m,k] * B[k,n]; grid (ceil(N/TN), ceil(M/TM), B*H); 256 threads, 4x4 per thread.
__global__ void __launch_bounds__(256)
sgemm_strided_kernel(const float* __restrict__ A, Mat la, const float* __restrict__ Bm, Mat lb,
                     float* __restrict__ C, Mat lc, int M, int N, int K, int H, float alpha) {
  __shared__ float sA[TK][TM + 4];
  __shared__ float sB[TK][TN + 4];
  const int z = blockIdx.z, b = z / H, h = z % H;
  const float* Ap = A + b * la.sb + h * la.sh;
  const float* Bp = Bm + b * lb.sb + h * lb.sh;
  float* Cp = C + b * lc.sb + h * lc.sh;
  const int m0 = blockIdx.y * TM, n0 = blockIdx.x * TN;
  const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  const bool a_kfast = (la.sc == 1);   // A contiguous along k
  const bool b_kfast = (lb.sr == 1);   // B contiguous along k
  for (int k0 = 0; k0 < K; k0 += TK) {
    // ---- stage A tile (TM x TK) as sA[k][m]
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      const int e = threadIdx.x + it * 256;
      int m, k;
      if (a_kfast) { k = e % TK; m = e / TK; } else { m = e % TM; k = e / TM; }
      const int gm = m0 + m, gk = k0 + k;
      sA[k][m] = (gm < M && gk < K) ? __ldg(Ap + gm * la.sr + gk * la.sc) : 0.f;
    }
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      const int e = threadIdx.x + it * 256;
      int n, k;
      if (b_kfast) { k = e % TK; n = e / TK; } else { n = e % TN; k = e / TN; }
      const int gn = n0 + n, gk = k0 + k;
      sB[k][n] = (gn < N && gk < K) ? __ldg(Bp + gk * lb.sr + gn * lb.sc) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < TK; ++k) {
      float a[4], bb[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = sA[k][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) bb[j] = sB[k][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], bb[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int gm = m0 + ty * 4 + i;
    if (gm >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int gn = n0 + tx * 4 + j;
      if (gn < N) Cp[gm * lc.sr + gn * lc.sc] = alpha * acc[i][j];
    }
  }
}

}  // namespace

int acr::launch_sgemm(const float* A, Mat la, const float* B, Mat lb, float* C, Mat lc,
                      int M, int N, int K, int batch, int H, float alpha, cudaStream_t st) {
  dim3 grid((N + TN - 1) / TN, (M + TM - 1) / TM, batch * H);
  sgemm_strided_kernel<<<grid, 256, 0, st>>>(A, la, B, lb, C, lc, M, N, K, H, alpha);
  return acr::check_launch("sgemm_strided_kernel");
}

using acr::launch_sgemm;

namespace {

// In-place row softmax over rows of length N; one CTA per row.
__global__ void __launch_bounds__(256)
softmax_rows_kernel(float* __restrict__ P, int N) {
  __shared__ float red[32];
  float* row = P + (long long)blockIdx.x * N;
  float m = -INFINITY;
  for (int j = threadIdx.x; j < N; j += blockDim.x) m = fmaxf(m, row[j]);
  m = acr::block_max(m, red);
  float s = 0.f;
  for (int j = threadIdx.x; j < N; j += blockDim.x) {
    const float e = expf(row[j] - m);
    row[j] = e;
    s += e;
  }
  s = acr::block_sum(s, red);
  const float inv = 1.f / s;
  for (int j = threadIdx.x; j < N; j += blockDim.x) row[j] *= inv;
}

// mean[b,i,j] = (1/H) sum_h P[b,h,i,j]
__global__ void __launch_bounds__(256)
head_mean_kernel(const float* __restrict__ P, float* __restrict__ mean, long long mean_bs, int H, long long NN) {
  const int b = blockIdx.y;
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= NN) return;
  const float* p = P + (long long)b * H * NN + e;
  float s = 0.f;
  for (int h = 0; h < H; ++h) s += __ldg(p + h * NN);
  mean[b * mean_bs + e] = s / (float)H;
}

// dP <- dP + G/H (what the reference hook stores); dS = P * (dP - rowsum(P*dP)).  One CTA per (b,h,i) row.
__global__ void __launch_bounds__(256)
softmax_bwd_rows_kernel(const float* __restrict__ P, float* __restrict__ dP, float* __restrict__ dS,
                        const float* __restrict__ G, long long g_bs, int H, int N) {
  __shared__ float red[32];
  const long long r = blockIdx.x;            // (b*H + h)*N + i
  const int i = (int)(r % N);
  const int b = (int)(r / ((long long)N * H));
  const float* p = P + r * N;
  float* dp = dP + r * N;
  float* ds = dS + r * N;
  const float* g = G ? G + b * g_bs + (long long)i * N : nullptr;
  const float invH = 1.f / (float)H;
  float dot = 0.f;
  for (int j = threadIdx.x; j < N; j += blockDim.x) {
    float v = dp[j];
    if (g) { v += __ldg(g + j) * invH; dp[j] = v; }
    dot += p[j] * v;
  }
  dot = acr::block_sum(dot, red);
  for (int j = threadIdx.x; j < N; j += blockDim.x) ds[j] = p[j] * (dp[j] - dot);
}

}  // namespace

extern "C" int acr_attn_fwd_f32(const float* qkv, int B, int N, int H, int D, float scale,
                                float* P, float* out,
                                float* attn_mean, long long mean_batch_stride, void* stream) {
  ACR_REQUIRE(qkv && P && out, ACR_E_INVAL, "acr_attn_fwd_f32: null pointer");
  ACR_REQUIRE(B > 0 && N > 0 && H > 0 && D > 0, ACR_E_INVAL, "acr_attn_fwd_f32: bad shape");
  ACR_REQUIRE((long long)B * H * N < (1ll << 31) && (long long)B * H <= 65535, ACR_E_INVAL, "acr_attn_fwd_f32: batch too large");
  ACR_REQUIRE(attn_mean == nullptr || (mean_batch_stride >= 0 && (B == 1 || mean_batch_stride >= (long long)N * N)), ACR_E_INVAL,
              "acr_attn_fwd_f32: mean_batch_stride %lld < N*N: the images' maps would overlap", mean_batch_stride);
  cudaStream_t st = (cudaStream_t)stream;
  const long long E = (long long)H * D, E3 = 3 * E, NN = (long long)N * N;
  const Mat lq{N * E3, D, E3, 1};                 // Q(i,d)
  const Mat lkT{N * E3, D, 1, E3};                // K^T(d,j)
  const Mat lp{H * NN, NN, N, 1};                 // P(i,j)
  if (int e = launch_sgemm(qkv, lq, qkv + E, lkT, P, lp, N, N, D, B, H, scale, st)) return e;
  softmax_rows_kernel<<<(unsigned)((long long)B * H * N), 256, 0, st>>>(P, N);
  if (int e = acr::check_launch("softmax_rows_kernel")) return e;
  const Mat lv{N * E3, D, E3, 1};                 // V(j,d)
  const Mat lo{N * E, D, E, 1};                   // out(i,d) inside [B,N,H*D]
  if (int e = launch_sgemm(P, lp, qkv + 2 * E, lv, out, lo, N, D, N, B, H, 1.f, st)) return e;
  if (attn_mean) {
    dim3 grid((unsigned)((NN + 255) / 256), B);
    head_mean_kernel<<<grid, 256, 0, st>>>(P, attn_mean, mean_batch_stride, H, NN);
    if (int e = acr::check_launch("head_mean_kernel")) return e;
  }
  return 0;
}

extern "C" int acr_attn_bwd_f32(const float* qkv, const float* P, const float* d_out,
                                int B, int N, int H, int D, float scale,
                                const float* g_mean, long long g_batch_stride,
                                float* dP, float* dS, float* d_qkv, void* stream) {
  ACR_REQUIRE(qkv && P && d_out && dP && dS && d_qkv, ACR_E_INVAL, "acr_attn_bwd_f32: null pointer");
  ACR_REQUIRE(B > 0 && N > 0 && H > 0 && D > 0, ACR_E_INVAL, "acr_attn_bwd_f32: bad shape");
  ACR_REQUIRE((long long)B * H * N < (1ll << 31) && (long long)B * H <= 65535, ACR_E_INVAL, "acr_attn_bwd_f32: batch too large");
  cudaStream_t st = (cudaStream_t)stream;
  const long long E = (long long)H * D, E3 = 3 * E, NN = (long long)N * N;
  const Mat lp{H * NN, NN, N, 1};                 // P / dP / dS (i,j)
  const Mat lpT{H * NN, NN, 1, N};                // transposed view (j,i)
  const Mat ldo{N * E, D, E, 1};                  // dO(i,d)
  const Mat lvT{N * E3, D, 1, E3};                // V^T(d,j)
  const Mat lx{N * E3, D, E3, 1};                 // Q/K/V (n,d) and dQ/dK/dV
  // dP = dO V^T
  if (int e = launch_sgemm(d_out, ldo, qkv + 2 * E, lvT, dP, lp, N, N, D, B, H, 1.f, st)) return e;
  softmax_bwd_rows_kernel<<<(unsigned)((long long)B * H * N), 256, 0, st>>>(P, dP, dS, g_mean, g_batch_stride, H, N);
  if (int e = acr::check_launch("softmax_bwd_rows_kernel")) return e;
  // dV = P^T dO
  if (int e = launch_sgemm(P, lpT, d_out, ldo, d_qkv + 2 * E, lx, N, D, N, B, H, 1.f, st)) return e;
  // dQ = scale * dS K
  if (int e = launch_sgemm(dS, lp, qkv + E, lx, d_qkv, lx, N, D, N, B, H, scale, st)) return e;
  // dK = scale * dS^T Q
  if (int e = launch_sgemm(dS, lpT, qkv, lx, d_qkv + E, lx, N, D, N, B, H, scale, st)) return e;
  return 0;
}
