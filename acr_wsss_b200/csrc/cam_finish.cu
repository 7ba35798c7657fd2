// Finish of batched CAM inference (infer_cam.py:153-215 for a batch): every output plane of every image goes from the
// low-res maps of all scales to the original image size, flipped view included, summed and min-max normalised, in ONE launch.
//
// A plane = one present class of one image, as the GETAM map (cams_s, align_corners=True, eps 1e-6) or the patch CAM
// (patch_s times the label value, align_corners=False, eps 1e-5).  A thread-block CLUSTER of kCluster CTAs owns a plane;
// each CTA takes a band of rows:
//   1. stage the low-res rows its band samples, both views of every scale, in shared memory (a gather of one channel);
//   2. bilinear samples with ATen's upsample_bilinear2d arithmetic for an explicit output size, summed in the reference's
//      order (scales in order, flipped view first), written to the output; band min / max on the side;
//   3. min / max of the plane through distributed shared memory (exact, so independent of order);
//   4. every thread normalises the values it wrote itself: (x - min) / (max - min + eps).
// No atomics, no cross-CTA float sums: two calls give bitwise-identical output.
#include "common.cuh"
#include <cooperative_groups.h>

namespace cg = cooperative_groups;

namespace {

constexpr int kCluster = 8;          // CTAs per plane
constexpr int kThreads = 256;
constexpr int kMaxScales = 8;
constexpr int kPlaneWords = 6;       // {offset, image, channel, kind, rows, cols}
constexpr size_t kMaxSmem = 200 * 1024;

struct ScaleMaps {
  const float* cams;                 // [2M, ph*pw, n]
  const float* patch;                // [2M, ph*pw, C]
  int ph, pw;
};

struct Params {
  ScaleMaps sc[kMaxScales];
  int ns, M, n, C;
  const long long* planes;           // device copy of the plane table
  const float* labels;               // [M, C]
  float* out;
};

// One axis of ATen's upsample_bilinear2d (explicit output size): taps i0, i1 and weights l0, l1.  The source index is
// computed with explicit rounding so that the band's row range (thread 0) and the per-pixel taps agree exactly.
struct Tap {
  int i0, i1;
  float l0, l1;
};
__device__ __forceinline__ float axis_scale(int in, int out, bool align) {
  if (align) return out > 1 ? (float)(in - 1) / (float)(out - 1) : 0.f;
  return (float)in / (float)out;
}
__device__ __forceinline__ Tap axis_tap(int in, float scale, int dst, bool align) {
  float src = align ? __fmul_rn(scale, (float)dst) : __fmaf_rn(scale, (float)dst + 0.5f, -0.5f);
  if (!align && src < 0.f) src = 0.f;
  Tap t;
  t.i0 = (int)src;
  t.i1 = t.i0 + (t.i0 < in - 1 ? 1 : 0);
  t.l1 = src - (float)t.i0;
  t.l0 = 1.f - t.l1;
  return t;
}

__global__ void __cluster_dims__(kCluster, 1, 1) __launch_bounds__(kThreads)
cam_finish_kernel(const __grid_constant__ Params p) {
  extern __shared__ float lowres[];                    // per scale: [2 views][band's low-res rows][pw]
  __shared__ int s_lo[kMaxScales], s_nr[kMaxScales], s_base[kMaxScales];
  __shared__ float s_rscale[kMaxScales], s_cscale[kMaxScales];
  __shared__ float s_red[2][kThreads / 32];
  __shared__ float2 s_band;                            // this CTA's (min, max), read by the whole cluster
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  const long long* d = p.planes + (long long)blockIdx.y * kPlaneWords;
  const long long off = d[0];
  const int m = (int)d[1], ch = (int)d[2], rows = (int)d[4], cols = (int)d[5];
  const bool patch = d[3] == 1;
  const bool align = !patch;
  const int r0 = (int)((long long)rows * rank / kCluster), r1 = (int)((long long)rows * (rank + 1) / kCluster);

  if (threadIdx.x == 0) {
    int base = 0;
    for (int s = 0; s < p.ns; ++s) {
      const int ph = p.sc[s].ph, pw = p.sc[s].pw;
      const float rs = axis_scale(ph, rows, align);
      int lo = 0, nr = 0;
      if (r1 > r0) {                                   // source rows are monotonic in the output row
        lo = axis_tap(ph, rs, r0, align).i0;
        nr = axis_tap(ph, rs, r1 - 1, align).i1 - lo + 1;
      }
      s_lo[s] = lo;
      s_nr[s] = nr;
      s_base[s] = base;
      s_rscale[s] = rs;
      s_cscale[s] = axis_scale(pw, cols, align);
      base += 2 * nr * pw;
    }
  }
  __syncthreads();
  for (int s = 0; s < p.ns; ++s) {
    const int pw = p.sc[s].pw, np = p.sc[s].ph * pw, nr = s_nr[s];
    const float* src = patch ? p.sc[s].patch : p.sc[s].cams;
    const int stride = patch ? p.C : p.n;
    float* dst = lowres + s_base[s];
    for (int i = threadIdx.x; i < 2 * nr * pw; i += kThreads) {
      const int v = i / (nr * pw), rem = i - v * nr * pw;
      const long long pix = (long long)(v * p.M + m) * np + (long long)(s_lo[s] + rem / pw) * pw + rem % pw;
      dst[i] = __ldg(src + pix * stride + ch);
    }
  }
  __syncthreads();

  const float label = patch ? __ldg(p.labels + (long long)m * p.C + ch) : 1.f;
  float* plane = p.out + off;
  float mn = INFINITY, mx = -INFINITY;
  for (int r = r0 + warp; r < r1; r += kThreads / 32) {
    Tap th[kMaxScales];                                // row taps, relative to the staged rows of view 0
#pragma unroll
    for (int s = 0; s < kMaxScales; ++s)
      if (s < p.ns) {
        th[s] = axis_tap(p.sc[s].ph, s_rscale[s], r, align);
        th[s].i0 = s_base[s] + (th[s].i0 - s_lo[s]) * p.sc[s].pw;
        th[s].i1 = s_base[s] + (th[s].i1 - s_lo[s]) * p.sc[s].pw;
      }
    for (int c = lane; c < cols; c += 32) {
      float acc = 0.f;
#pragma unroll
      for (int s = 0; s < kMaxScales; ++s)
        if (s < p.ns) {
          const int pw = p.sc[s].pw, vstride = s_nr[s] * pw;
#pragma unroll
          for (int v = 0; v < 2; ++v) {                // view 0 is the flipped input: output column c samples column cols-1-c
            const Tap tw = axis_tap(pw, s_cscale[s], v == 0 ? cols - 1 - c : c, align);
            const float* a = lowres + th[s].i0 + v * vstride;
            const float* b = lowres + th[s].i1 + v * vstride;
            float val = th[s].l0 * (tw.l0 * a[tw.i0] + tw.l1 * a[tw.i1]) + th[s].l1 * (tw.l0 * b[tw.i0] + tw.l1 * b[tw.i1]);
            if (patch) val = __fmul_rn(val, label);   // the reference rounds the product before the sum
            acc += val;
          }
        }
      plane[(long long)r * cols + c] = acc;
      mn = fminf(mn, acc);
      mx = fmaxf(mx, acc);
    }
  }
  mn = -acr::warp_max(-mn);
  mx = acr::warp_max(mx);
  if (lane == 0) {
    s_red[0][warp] = mn;
    s_red[1][warp] = mx;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < kThreads / 32; ++w) {
      mn = fminf(mn, s_red[0][w]);
      mx = fmaxf(mx, s_red[1][w]);
    }
    s_band = make_float2(mn, mx);
  }
  cluster.sync();
  mn = INFINITY;
  mx = -INFINITY;
  for (int q = 0; q < kCluster; ++q) {
    const float2 b = *cluster.map_shared_rank(&s_band, q);
    mn = fminf(mn, b.x);
    mx = fmaxf(mx, b.y);
  }
  cluster.sync();                                      // nobody leaves while its (min, max) is still being read
  const float den = (mx - mn) + (patch ? 1e-5f : 1e-6f);
  for (int r = r0 + warp; r < r1; r += kThreads / 32)
    for (int c = lane; c < cols; c += 32) {
      float* q = plane + (long long)r * cols + c;      // written by this thread above
      *q = (*q - mn) / den;
    }
}

}  // namespace

extern "C" int acr_cam_finish(const float* const* cams_host, const float* const* patch_host, const int* grid_host, int num_scales,
                              int M, int n, int C, const float* labels, const long long* planes_host, int num_planes,
                              float* out, long long out_elems, void* workspace, size_t workspace_bytes, void* stream) {
  ACR_REQUIRE(cams_host && patch_host && grid_host && labels, ACR_E_INVAL, "acr_cam_finish: null pointer");
  ACR_REQUIRE(num_scales >= 1 && num_scales <= kMaxScales, ACR_E_INVAL, "acr_cam_finish: %d scales (1..%d)", num_scales, kMaxScales);
  ACR_REQUIRE(M >= 1 && n >= 1 && C >= 1, ACR_E_INVAL, "acr_cam_finish: bad shape M=%d n=%d C=%d", M, n, C);
  ACR_REQUIRE(num_planes >= 0 && num_planes <= 65535, ACR_E_INVAL, "acr_cam_finish: %d planes (0..65535)", num_planes);
  ACR_REQUIRE(num_planes == 0 || (planes_host && out && workspace), ACR_E_INVAL, "acr_cam_finish: null pointer");
  Params p = {};
  p.ns = num_scales; p.M = M; p.n = n; p.C = C;
  size_t smem = 0;
  for (int s = 0; s < num_scales; ++s) {
    ACR_REQUIRE(cams_host[s] && patch_host[s], ACR_E_INVAL, "acr_cam_finish: null map pointer at scale %d", s);
    const int ph = grid_host[2 * s], pw = grid_host[2 * s + 1];
    ACR_REQUIRE(ph >= 1 && pw >= 1, ACR_E_INVAL, "acr_cam_finish: bad grid %dx%d at scale %d", ph, pw, s);
    p.sc[s] = {cams_host[s], patch_host[s], ph, pw};
    smem += 2 * (size_t)ph * pw * sizeof(float);
  }
  ACR_REQUIRE(smem <= kMaxSmem, ACR_E_INVAL, "acr_cam_finish: low-res maps of %zu bytes exceed %zu bytes of shared memory", smem, kMaxSmem);
  for (int i = 0; i < num_planes; ++i) {
    const long long* d = planes_host + (long long)i * kPlaneWords;
    const long long offset = d[0], image = d[1], channel = d[2], kind = d[3], rows = d[4], cols = d[5];
    ACR_REQUIRE(image >= 0 && image < M && (kind == 0 || kind == 1) && channel >= 0 && channel < (kind == 0 ? n : C),
                ACR_E_INVAL, "acr_cam_finish: plane %d: bad image / kind / channel", i);
    ACR_REQUIRE(rows >= 1 && cols >= 1 && rows <= INT32_MAX && cols <= INT32_MAX, ACR_E_INVAL, "acr_cam_finish: plane %d: bad size", i);
    ACR_REQUIRE(offset >= 0 && offset <= out_elems && rows <= (out_elems - offset) / cols, ACR_E_INVAL,
                "acr_cam_finish: plane %d overflows the %lld-element output", i, out_elems);
  }
  const size_t table = (size_t)num_planes * kPlaneWords * sizeof(long long);
  ACR_REQUIRE(workspace_bytes >= table, ACR_E_NOMEM, "acr_cam_finish: workspace of %zu bytes needed", table);
  ACR_REQUIRE(((uintptr_t)workspace & 7) == 0, ACR_E_ALIGN, "acr_cam_finish: workspace must be 8-byte aligned");
  if (num_planes == 0) return 0;
  ACR_REQUIRE(acr_device_is_sm100(), ACR_E_NOSM100, "acr_cam_finish: needs an sm_100 device");
  const cudaStream_t st = (cudaStream_t)stream;
  ACR_CUDA(cudaMemcpyAsync(workspace, planes_host, table, cudaMemcpyHostToDevice, st));
  p.planes = (const long long*)workspace;
  p.labels = labels;
  p.out = out;
  static bool attr_set[64] = {false};
  if (smem > 48 * 1024) {
    int dev = 0;
    ACR_CUDA(cudaGetDevice(&dev));
    if (!(dev >= 0 && dev < 64 && attr_set[dev])) {
      ACR_CUDA(cudaFuncSetAttribute(cam_finish_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
      if (dev >= 0 && dev < 64) attr_set[dev] = true;
    }
  }
  acr::KernelTimer kt_("cam_finish_kernel", st);
  cam_finish_kernel<<<dim3(kCluster, num_planes), kThreads, smem, st>>>(p);
  return acr::check_launch("cam_finish_kernel");
}
