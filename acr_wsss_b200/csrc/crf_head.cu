// Head of the dense-CRF regulariser (BASELINE configs[3], train_acr_coco.py + myTool.py:825-857 call shape): the probabilities the
// bilateral filter is applied to.  What the step computes from the patch-token logits z [B, P*P, C] (channel-last, as
// cls_head produces them for layer_4[:,1:]):
//     up   = bilinear(z -> S x S, align_corners=False)                       [B, C, S, S]
//     prob = softmax over [0 (background), up_1 .. up_C]                     [B, C+1, S, S]
//     seg  = bilinear(prob -> S/2 x S/2, align_corners=False, scale 0.5)     [B, C+1, S/2, S/2]   (= the 2x2 mean)
// As library calls this is six elementwise passes over 0.5 GB tensors per step at 448x448, C = 80 (forward and backward): 24 of
// the 37.6 ms of the COCO-shaped step.  Here the full-resolution tensors never exist in the forward (one thread per output pixel
// interpolates, normalises and averages its four source pixels from the L1-resident patch logits); the backward recomputes the
// softmax per full-resolution pixel and emits d(up) once, which bilinear_up_bwd_kernel (gather form, no atomics) folds to patch resolution.
// The interpolation follows ATen's upsample_bilinear2d (source index scale*(dst+0.5)-0.5 clamped at 0, lambda order of its kernel).
#include "common.cuh"

namespace {

struct Tap { int i0, i1; float l0, l1; };   // source rows (or columns) and their weights

__device__ __forceinline__ Tap make_tap(int dst, float scale, int n_in) {
  float src = scale * ((float)dst + 0.5f) - 0.5f;
  src = src < 0.f ? 0.f : src;
  Tap t;
  t.i0 = (int)src;
  if (t.i0 > n_in - 1) t.i0 = n_in - 1;
  t.i1 = t.i0 + (t.i0 < n_in - 1 ? 1 : 0);
  t.l1 = src - (float)t.i0;
  t.l0 = 1.f - t.l1;
  return t;
}

// interpolated logit of class c at a full-resolution pixel whose four source patches start at p00..p11 (rows of C floats)
__device__ __forceinline__ float interp(const float* p00, const float* p01, const float* p10, const float* p11, const Tap& ty, const Tap& tx, int c) {
  return ty.l0 * (tx.l0 * __ldg(p00 + c) + tx.l1 * __ldg(p01 + c)) + ty.l1 * (tx.l0 * __ldg(p10 + c) + tx.l1 * __ldg(p11 + c));
}

// The four full-resolution pixels (2y+dy, 2x+dx) behind one output pixel.  With an even up-sampling ratio (16 in the model) they
// interpolate between the SAME four patches and differ only in the tap weights, so one thread serves all four from one set of
// patch-row loads per class (16 FMAs for the four interpolated logits instead of 4 x (4 loads + 7)).  `shared` is false for ratios
// where a 2x2 group straddles a patch-centre line; each pixel then reads its own rows.
struct Quad {
  const float* p[4][4];     // [pixel][00, 01, 10, 11]
  Tap ty[2], tx[2];
  bool shared;
  float m[4], inv_s[4];
};

__device__ __forceinline__ void quad_logits(const Quad& q, int c, float (&l)[4]) {
  if (q.shared) {
    const float v00 = __ldg(q.p[0][0] + c), v01 = __ldg(q.p[0][1] + c), v10 = __ldg(q.p[0][2] + c), v11 = __ldg(q.p[0][3] + c);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const Tap& ty = q.ty[u >> 1];
      const Tap& tx = q.tx[u & 1];
      l[u] = ty.l0 * (tx.l0 * v00 + tx.l1 * v01) + ty.l1 * (tx.l0 * v10 + tx.l1 * v11);
    }
  } else {
#pragma unroll
    for (int u = 0; u < 4; ++u) l[u] = interp(q.p[u][0], q.p[u][1], q.p[u][2], q.p[u][3], q.ty[u >> 1], q.tx[u & 1], c);
  }
}

__device__ __forceinline__ void quad_setup(Quad& q, const float* zb, int y, int x, int P, int C, float scale) {
  q.ty[0] = make_tap(2 * y, scale, P); q.ty[1] = make_tap(2 * y + 1, scale, P);
  q.tx[0] = make_tap(2 * x, scale, P); q.tx[1] = make_tap(2 * x + 1, scale, P);
  q.shared = q.ty[0].i0 == q.ty[1].i0 && q.ty[0].i1 == q.ty[1].i1 && q.tx[0].i0 == q.tx[1].i0 && q.tx[0].i1 == q.tx[1].i1;
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const Tap& ty = q.ty[u >> 1];
    const Tap& tx = q.tx[u & 1];
    q.p[u][0] = zb + ((long long)ty.i0 * P + tx.i0) * C;
    q.p[u][1] = zb + ((long long)ty.i0 * P + tx.i1) * C;
    q.p[u][2] = zb + ((long long)ty.i1 * P + tx.i0) * C;
    q.p[u][3] = zb + ((long long)ty.i1 * P + tx.i1) * C;
  }
  // online max / sum over [0, up_1..up_C] of each of the four pixels (the background logit is the constant 0)
  float m[4] = {0.f, 0.f, 0.f, 0.f}, s[4] = {1.f, 1.f, 1.f, 1.f};
  for (int c = 0; c < C; ++c) {
    float l[4];
    quad_logits(q, c, l);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const float nm = fmaxf(m[u], l[u]);
      s[u] = s[u] * __expf(m[u] - nm) + __expf(l[u] - nm);
      m[u] = nm;
    }
  }
#pragma unroll
  for (int u = 0; u < 4; ++u) { q.m[u] = m[u]; q.inv_s[u] = 1.f / s[u]; }
}

// seg[b,k,y,x] = mean over the 2x2 full-resolution pixels of softmax_k.  One thread per (b,y,x).
__global__ void __launch_bounds__(128)
crf_head_fwd_kernel(const float* __restrict__ z, int P, int C, int S, float scale, float* __restrict__ seg) {
  const int h = S / 2;
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y, b = blockIdx.z;
  if (x >= h) return;
  Quad q;
  quad_setup(q, z + (long long)b * P * P * C, y, x, P, C, scale);
  float* out = seg + ((long long)b * (C + 1) * h + y) * h + x;
  const long long plane = (long long)h * h;
  float bg = 0.f;
#pragma unroll
  for (int u = 0; u < 4; ++u) bg += __expf(-q.m[u]) * q.inv_s[u];
  out[0] = 0.25f * bg;
  for (int c = 0; c < C; ++c) {
    float l[4];
    quad_logits(q, c, l);
    float acc = 0.f;
#pragma unroll
    for (int u = 0; u < 4; ++u) acc += __expf(l[u] - q.m[u]) * q.inv_s[u];
    out[(long long)(c + 1) * plane] = 0.25f * acc;
  }
}

// d_up[b,c,Y,X] = p_c * (g_c - sum_j p_j g_j) with p = softmax at the full-resolution pixel and g = 0.25 * g_seg[b,:,Y/2,X/2]
// (the 2x2 mean gives every source pixel a quarter of the output gradient).  One thread per OUTPUT pixel (b,y,x): its four
// full-resolution pixels share the gradient row g and (see Quad) the patch rows; results leave as two 8-byte stores per class.
__global__ void __launch_bounds__(128)
crf_head_bwd_kernel(const float* __restrict__ z, const float* __restrict__ g_seg, int P, int C, int S, float scale, float* __restrict__ d_up) {
  const int h = S / 2;
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y, b = blockIdx.z;
  if (x >= h) return;
  Quad q;
  quad_setup(q, z + (long long)b * P * P * C, y, x, P, C, scale);
  const long long plane = (long long)h * h;
  const float* g = g_seg + ((long long)b * (C + 1) * h + y) * h + x;
  const float g0 = __ldg(g);
  float t[4];
#pragma unroll
  for (int u = 0; u < 4; ++u) t[u] = __expf(-q.m[u]) * q.inv_s[u] * g0;      // background term of sum_j p_j g_j
  for (int c = 0; c < C; ++c) {
    float l[4];
    quad_logits(q, c, l);
    const float gc = __ldg(g + (long long)(c + 1) * plane);
#pragma unroll
    for (int u = 0; u < 4; ++u) t[u] += __expf(l[u] - q.m[u]) * q.inv_s[u] * gc;
  }
  float* out = d_up + ((long long)b * C * S + 2 * y) * S + 2 * x;      // S even: (2y, 2x) is 8-byte aligned
  const long long oplane = (long long)S * S;
  for (int c = 0; c < C; ++c) {
    float l[4], d[4];
    quad_logits(q, c, l);
    const float gc = __ldg(g + (long long)(c + 1) * plane);
#pragma unroll
    for (int u = 0; u < 4; ++u) d[u] = 0.25f * __expf(l[u] - q.m[u]) * q.inv_s[u] * (gc - t[u]);
    *reinterpret_cast<float2*>(out + (long long)c * oplane) = make_float2(d[0], d[1]);
    *reinterpret_cast<float2*>(out + (long long)c * oplane + S) = make_float2(d[2], d[3]);
  }
}

// Backward of the bilinear up-sampling (align_corners=False): d_patch[b,c,py,px] = sum_{Y,X} wy(Y,py) wx(X,px) d_up[b,c,Y,X].
// (ATen's upsample_bilinear2d_backward scatters with one atomic per output pixel and tap: 16.6 ms for [8,80,448,448].)
// One CTA per (b,c) plane, one thread per four columns (128-bit loads) walking the rows once.  Rows with the same upper source row i0 form a group;
// when a group ends, patch row py = i0 has all its contributions (weight l0 from this group, l1 from the previous one), the
// column sums go to shared memory and 16 lanes per patch column fold them with the column weights.
constexpr int kUpBwdThreads = 128, kUpBwdMaxS = 4 * kUpBwdThreads;
__global__ void __launch_bounds__(kUpBwdThreads)
bilinear_up_bwd_kernel(const float* __restrict__ d_up, int P, int S, float scale, float* __restrict__ d_patch) {
  // shared: column sums [kUpBwdMaxS], the tap table of a row / column index (i0, l1: the image is square) [S], per patch column
  // the range of up-sampled columns that touch it [P]
  extern __shared__ float sm[];
  float* colsum = sm;
  int* t_i0 = reinterpret_cast<int*>(sm + kUpBwdMaxS);
  float* t_l1 = reinterpret_cast<float*>(t_i0 + S);
  int* x_lo = reinterpret_cast<int*>(t_l1 + S);
  int* x_hi = x_lo + P;
  for (int i = threadIdx.x; i < S; i += kUpBwdThreads) {
    const Tap t = make_tap(i, scale, P);
    t_i0[i] = t.i0;
    t_l1[i] = t.l1;
  }
  __syncthreads();
  for (int px = threadIdx.x; px < P; px += kUpBwdThreads) {      // columns with i0 in {px - 1, px} (i0 is non-decreasing)
    int lo = 0;
    while (lo < S && t_i0[lo] < px - 1) ++lo;
    int hi = lo;
    while (hi < S && t_i0[hi] <= px) ++hi;
    x_lo[px] = lo;
    x_hi[px] = hi;
  }
  const float* plane = d_up + (size_t)blockIdx.x * S * S;
  float* outp = d_patch + (size_t)blockIdx.x * P * P;
  const int X0 = 4 * threadIdx.x;               // this thread's four columns
  const bool vec = (S & 3) == 0;
  float4 carry = make_float4(0.f, 0.f, 0.f, 0.f);
  int Y = 0;
  while (Y < S) {
    const int g = t_i0[Y];
    int Yend = Y + 1;
    while (Yend < S && t_i0[Yend] == g) ++Yend;
    const bool last = g >= P - 1;               // i1 == i0: both weights go to patch row g
    float4 a0 = carry, a1 = make_float4(0.f, 0.f, 0.f, 0.f);
    if (X0 < S) {
#pragma unroll 4
      for (int yy = Y; yy < Yend; ++yy) {
        const float l1 = t_l1[yy], l0 = 1.f - l1;
        float4 v;
        const float* src = plane + (size_t)yy * S + X0;
        if (vec) {
          v = __ldg(reinterpret_cast<const float4*>(src));
        } else {
          v.x = __ldg(src);
          v.y = X0 + 1 < S ? __ldg(src + 1) : 0.f;
          v.z = X0 + 2 < S ? __ldg(src + 2) : 0.f;
          v.w = X0 + 3 < S ? __ldg(src + 3) : 0.f;
        }
        const float w0 = last ? 1.f : l0;       // (l0 + l1 = 1)
        a0.x = fmaf(w0, v.x, a0.x); a0.y = fmaf(w0, v.y, a0.y); a0.z = fmaf(w0, v.z, a0.z); a0.w = fmaf(w0, v.w, a0.w);
        if (!last) { a1.x = fmaf(l1, v.x, a1.x); a1.y = fmaf(l1, v.y, a1.y); a1.z = fmaf(l1, v.z, a1.z); a1.w = fmaf(l1, v.w, a1.w); }
      }
      *reinterpret_cast<float4*>(colsum + X0) = a0;
    }
    carry = a1;
    Y = Yend;
    __syncthreads();
    // patch row g: 16 lanes per patch column fold the column sums of its ~2 S/P source columns
    for (int pxb = (threadIdx.x >> 5) * 2; pxb < P; pxb += (kUpBwdThreads >> 5) * 2) {      // warp-uniform trip count (shuffles below)
      const int px = pxb + ((threadIdx.x >> 4) & 1);
      float acc = 0.f;
      if (px < P) {
        for (int xx = x_lo[px] + (threadIdx.x & 15); xx < x_hi[px]; xx += 16) {
          const int i0 = t_i0[xx];
          const float l1 = t_l1[xx];
          const int i1 = i0 + (i0 < P - 1 ? 1 : 0);
          const float w = (i0 == px ? 1.f - l1 : 0.f) + (i1 == px ? l1 : 0.f);
          acc = fmaf(w, colsum[xx], acc);
        }
      }
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o, 16);
      if ((threadIdx.x & 15) == 0 && px < P) outp[g * P + px] = acc;
    }
    __syncthreads();
  }
}

}  // namespace

extern "C" int acr_bilinear_up_bwd(const float* d_up, int planes, int P, int S, float* d_patch, void* stream) {
  ACR_REQUIRE(d_up && d_patch, ACR_E_INVAL, "acr_bilinear_up_bwd: null pointer");
  ACR_REQUIRE(planes > 0 && P > 0 && S >= P && S <= kUpBwdMaxS, ACR_E_INVAL, "acr_bilinear_up_bwd: bad shape (P <= S <= %d)", kUpBwdMaxS);
  ACR_REQUIRE(((uintptr_t)d_up & 15) == 0, ACR_E_ALIGN, "acr_bilinear_up_bwd: d_up must be 16-byte aligned");
  const size_t smem = (size_t)(kUpBwdMaxS + 2 * S + 2 * P) * sizeof(float);
  bilinear_up_bwd_kernel<<<planes, kUpBwdThreads, smem, (cudaStream_t)stream>>>(d_up, P, S, (float)P / (float)S, d_patch);
  return acr::check_launch("bilinear_up_bwd_kernel");
}

extern "C" int acr_crf_head_fwd(const float* logits, int B, int P, int C, int S, float* seg, void* stream) {
  ACR_REQUIRE(logits && seg, ACR_E_INVAL, "acr_crf_head_fwd: null pointer");
  ACR_REQUIRE(B > 0 && B <= 65535 && P > 0 && P <= S && C > 0 && S >= 2 && (S % 2) == 0 && S / 2 <= 65535, ACR_E_INVAL,
              "acr_crf_head_fwd: bad shape (S even, P <= S)");
  const int h = S / 2;
  crf_head_fwd_kernel<<<dim3((h + 127) / 128, h, B), 128, 0, (cudaStream_t)stream>>>(logits, P, C, S, (float)P / (float)S, seg);
  return acr::check_launch("crf_head_fwd_kernel");
}

extern "C" int acr_crf_head_bwd(const float* logits, const float* g_seg, int B, int P, int C, int S, float* d_up, void* stream) {
  ACR_REQUIRE(logits && g_seg && d_up, ACR_E_INVAL, "acr_crf_head_bwd: null pointer");
  ACR_REQUIRE(B > 0 && B <= 65535 && P > 0 && P <= S && C > 0 && S >= 2 && (S % 2) == 0 && S <= 65535, ACR_E_INVAL,
              "acr_crf_head_bwd: bad shape (S even, P <= S)");
  const int h = S / 2;
  crf_head_bwd_kernel<<<dim3((h + 127) / 128, h, B), 128, 0, (cudaStream_t)stream>>>(logits, g_seg, P, C, S, (float)P / (float)S, d_up);
  return acr::check_launch("crf_head_bwd_kernel");
}
