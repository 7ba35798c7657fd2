// (a11) Permutohedral-lattice bilateral filter on the GPU.
// Reference: wrapper/bilateralfilter/bilateralfilter.cpp:4-55 (feature build, per-image / per-plane loop)
// and permutohedral.cpp:115-440 (Permutohedral::init, SSE branch) / :507-631 (Permutohedral::compute).
//
// What must match the reference (it is a lattice APPROXIMATION of a 5-D Gaussian, not an exact one):
//   * features (x/sxy, y/sxy, r/srgb, g/srgb, b/srgb), d = 5 (bilateralfilter.cpp:8-16);
//   * elevation with scale_i = (d+1)sqrt(2/3)/sqrt((i+1)(i+2)) by the running-sum recurrence (:339-345),
//     separate multiply and add roundings (the SSE code has no FMA -> __fmul_rn/__fadd_rn here);
//   * nearest-EVEN rounding to the remainder-0 simplex (:349-357, _mm_round_ps / cvtps) -> rintf;
//   * rank by pairwise comparison, sum fix-up (:359-380), barycentric weights in the same accumulation
//     order (:383-403), the d+1 vertex keys rem0 + canonical[remainder][rank] (:404-413);
//   * blur: for axis j = 0..d sequentially new = old + 0.5 (old[n1] + old[n2]) with n1/n2 = key -/+ 1 on all
//     coordinates and +/- d on coordinate j, missing neighbour = 0 (:423-436, :548-566);
//   * slice with alpha = 1/(1+2^-d), no normalisation (:567-583).
// What is free: vertex numbering and hash function (results are indexed by key, not by id), the order of
// the splat additions (float atomics here; differences are ~1e-7 relative), and filtering all K planes in one
// pass (the planes are independent and the filter is linear; the reference loops K times with value_size=1).
//
// Eleven launches per batch of up to 8 images (grid.z = image); round 1 needed 13 launches + 16 memsets and 450 us at N = 8, K = 21:
//   embed      per pixel: 6 candidate keys + barycentric weights, written plane-major (candidate c = r*HWp + pixel, so every
//              store is coalesced); the same threads clear the hash table and the vertex counter
//   insert     per candidate; neighbouring pixels mostly fall on the same lattice vertex, so a warp first groups its lanes by
//              key (__match_any_sync on a 32-bit hash, verified against the group leader's key) and only leaders probe the table
//   prepare    one persistent launch for three independent jobs: blur neighbours of every vertex (2 table lookups per
//              (vertex, axis)), candidate -> vertex id + 1, zeroing of the value arrays
//   splat      a CTA sorts the 768 (pixel, remainder) pairs of its 16 x 8 pixel block by vertex in shared memory (integer atomics
//              only) and issues ONE red.global.add.v4.f32 per (vertex, 4 planes) (K padded to a multiple of 4: 16-byte value rows)
//   blur       d+1 passes, one launch each, (vertex, 4 planes) items with 4 independent gather chains per thread
//   slice      per (pixel, 4 planes): six 128-bit gathers, same accumulation order as the reference
//
// Embedding, insertion, blur neighbours, slice and the data layout in HBM: lattice.cuh (D = 5, Pad = true).
#include "lattice.cuh"
#include <cmath>
#include <mutex>
#include <vector>

namespace {

using namespace acr::lattice;
constexpr int D5 = 5;          // feature dimension
constexpr int D6 = D5 + 1;
using Lat = Lattice<D5>;

// Steps 1-3 (lattice.cuh): the reference's SSE embedding with its phantom pads.
__global__ void __launch_bounds__(256)
lattice_embed_kernel(const float* __restrict__ image, int H, int W, float sigmargb, float sigmaxy, Scales<D5> sc, Lat lat0) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  embed<D5, true>(for_image(lat0, blockIdx.z), image + (size_t)blockIdx.z * 3 * H * W, H, W, sigmargb, sigmaxy, sc, idx,
                  gridDim.x * blockDim.x);
}

__global__ void __launch_bounds__(256)
lattice_insert_kernel(Lat lat0) {
  insert(for_image(lat0, blockIdx.z), blockIdx.x * blockDim.x + threadIdx.x);
}

// Step 3 plus the zero-fill of the value arrays (val0 entirely, slot 0 of val1).  The table lookups are latency bound: the
// second launch bound keeps 8 CTAs (full occupancy) per SM.
__global__ void __launch_bounds__(256, 8)
lattice_prepare_kernel(Lat lat0) {
  const Lat lat = for_image(lat0, blockIdx.z);
  const int nthreads = gridDim.x * blockDim.x, t0 = blockIdx.x * blockDim.x + threadIdx.x;
  prepare(lat, t0, nthreads);
  const long long nz = ((long long)*lat.counter + 1) * lat.Kp / 4;
  float4* z0 = reinterpret_cast<float4*>(lat.val0);
  for (long long i = t0; i < nz; i += nthreads) z0[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  if (t0 < lat.Kp) lat.val1[t0] = 0.f;
}

__device__ __forceinline__ void red_add_v4(float* addr, const float4& v) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

constexpr int kPixTile = 128;      // pixels per CTA (splat: 16 x 8 block of the image; slice: 128 consecutive pixels)
constexpr int kTileW = 16, kTileH = 8;
constexpr int kSlotProbes = 32;

// Splat.  A CTA owns a 16 x 8 block of pixels: its 768 (pixel, remainder) pairs fall on ~100-200 distinct lattice vertices.  Float
// atomics at L2 bounded the first version (50 M of them for N = 8, K = 21), and shared-memory float atomics are CAS loops (4x
// slower still, measured), so the pairs are SORTED by vertex inside the CTA with integer shared-memory atomics only:
//   1. input planes -> shared memory, transposed to tile4[pixel][quad] (float4 = 4 consecutive planes; odd row stride);
//   2. every pair finds its vertex's slot in a small open-addressing table (atomicCAS) and draws a position in the slot (atomicAdd);
//   3. exclusive scan of the slot counts, pairs scattered to order[] (counting sort);
//   4. one work item per (occupied slot, quad) sums its pairs from the tile and issues ONE red.global.add.v4.f32.
// Pairs that find no slot within kSlotProbes probes add to global memory directly (rare).
constexpr int kSplatSlots = 1024;    // >= the 768 pairs of a tile, so the table never fills up; 4 slots per thread in the scan
__global__ void __launch_bounds__(256)
lattice_splat_kernel(const float* __restrict__ in, int K, int H, int W, int HWpad, Lat lat0) {
  extern __shared__ float4 smem4[];                    // tile4[kPixTile][Qs], then the int / float arrays below
  __shared__ int skey[kSplatSlots], scount[kSplatSlots], sstart[kSplatSlots], socc[kSplatSlots], warp_tot[8], warp_occ[8], n_occ;
  const Lat lat = for_image(lat0, blockIdx.z);
  const int HW = H * W, Kp = lat.Kp, Q = Kp / 4;
  in += (size_t)blockIdx.z * K * HW;
  const int Qs = Q | 1;                                 // odd row stride (in float4): conflict-free 128-bit stores
  int* slot = reinterpret_cast<int*>(smem4 + (size_t)Qs * kPixTile);      // [D6 * kPixTile]: slot of the pair, -1 = none
  int* pos = slot + D6 * kPixTile;                                        // position inside the slot
  int* order = pos + D6 * kPixTile;                                       // pair indices sorted by slot
  float* wts = reinterpret_cast<float*>(order + D6 * kPixTile);
  const int tiles_x = (W + kTileW - 1) / kTileW;
  const int x0 = (blockIdx.x % tiles_x) * kTileW, y0 = (blockIdx.x / tiles_x) * kTileH;
  for (int i = threadIdx.x; i < kSplatSlots; i += blockDim.x) { skey[i] = 0; scount[i] = 0; }
  for (int e = threadIdx.x; e < Q * kPixTile; e += blockDim.x) {      // four coalesced plane reads -> one 16-byte store
    const int q = e / kPixTile, p = e - q * kPixTile;
    const int x = x0 + (p % kTileW), y = y0 + (p / kTileW);
    float v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) v[j] = (4 * q + j < K && x < W && y < H) ? __ldg(in + (size_t)(4 * q + j) * HW + (size_t)y * W + x) : 0.f;
    smem4[p * Qs + q] = make_float4(v[0], v[1], v[2], v[3]);
  }
  __syncthreads();
  for (int w = threadIdx.x; w < D6 * kPixTile; w += blockDim.x) {
    const int p = w % kPixTile, r = w / kPixTile;
    const int x = x0 + (p % kTileW), y = y0 + (p / kTileW);
    int sl = -1;
    float wt = 0.f;
    if (x < W && y < H) {
      const int pix = y * W + x;
      const int o = __ldg(lat.offs + (size_t)r * HWpad + pix);
      wt = __ldg(lat.bary + (size_t)r * HWpad + pix);
      const uint32_t h = ((uint32_t)o * 0x9E3779B1u) >> 7;
      for (int t = 0; t < kSlotProbes; ++t) {
        const int i = (int)((h + t) & (uint32_t)(kSplatSlots - 1));
        const int prev = atomicCAS(&skey[i], 0, o);
        if (prev == 0 || prev == o) { sl = i; break; }
      }
      if (sl >= 0) {
        pos[w] = atomicAdd(&scount[sl], 1);
      } else {                                          // table neighbourhood full (rare): this pair adds to global memory itself
        for (int q = 0; q < Q; ++q) {
          const float4 x = smem4[p * Qs + q];
          red_add_v4(lat.val0 + (size_t)o * Kp + 4 * q, make_float4(wt * x.x, wt * x.y, wt * x.z, wt * x.w));
        }
      }
    }
    slot[w] = sl;
    wts[w] = wt;
  }
  __syncthreads();
  {   // exclusive scan of scount (4 consecutive slots per thread) and compaction of the occupied slots
    constexpr int PER = kSplatSlots / 256;
    const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
    int c[PER], tot = 0, occ = 0;
#pragma unroll
    for (int u = 0; u < PER; ++u) { c[u] = scount[threadIdx.x * PER + u]; tot += c[u]; occ += c[u] > 0; }
    int v = tot, vo = occ;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int n = __shfl_up_sync(0xffffffffu, v, o), no = __shfl_up_sync(0xffffffffu, vo, o);
      if (lane >= o) { v += n; vo += no; }
    }
    if (lane == 31) { warp_tot[wp] = v; warp_occ[wp] = vo; }
    __syncthreads();
    int base = v - tot, obase = vo - occ;
    for (int i = 0; i < wp; ++i) { base += warp_tot[i]; obase += warp_occ[i]; }
#pragma unroll
    for (int u = 0; u < PER; ++u) {
      sstart[threadIdx.x * PER + u] = base;
      base += c[u];
      if (c[u] > 0) socc[obase++] = threadIdx.x * PER + u;
    }
    if (threadIdx.x == blockDim.x - 1) n_occ = obase;
  }
  __syncthreads();
  for (int w = threadIdx.x; w < D6 * kPixTile; w += blockDim.x) {
    const int sl = slot[w];
    if (sl >= 0) order[sstart[sl] + pos[w]] = w;
  }
  __syncthreads();
  const int nitems = n_occ * Q;
  for (int w = threadIdx.x; w < nitems; w += blockDim.x) {
    const int sidx = socc[w / Q], q = w % Q;
    const int beg = sstart[sidx], n = scount[sidx];
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int j = 0; j < n; ++j) {
      const int pw = order[beg + j];
      const float wt = wts[pw];
      const float4 x = smem4[(pw % kPixTile) * Qs + q];
      acc.x = fmaf(wt, x.x, acc.x); acc.y = fmaf(wt, x.y, acc.y); acc.z = fmaf(wt, x.z, acc.z); acc.w = fmaf(wt, x.w, acc.w);
    }
    red_add_v4(lat.val0 + (size_t)skey[sidx] * Kp + 4 * q, acc);
  }
}

// One blur pass along axis j: new = old + 0.5 * (old[n1] + old[n2]).  Work item = (vertex, 4 planes); the chain neighbour ids ->
// three gathers is pure L2 latency, so every thread keeps kBlurIlp independent items in flight.  One launch per pass over the whole
// GPU: a single launch with one 8-CTA cluster per image and cluster barriers between the passes was measured as well -- no faster
// on small lattices (75 vs 78 us at 15 k vertices) and 64 of 148 SMs wide on large ones (noise images: 300 k vertices per image).
constexpr int kBlurIlp = 4;
__global__ void __launch_bounds__(256)
lattice_blur_kernel(const float* __restrict__ old0, float* __restrict__ new0, int j, Lat lat0) {
  const Lat lat = for_image(lat0, blockIdx.z);
  const float* oldv = img_ptr(old0, lat.ws, blockIdx.z);
  float* newv = img_ptr(new0, lat.ws, blockIdx.z);
  const long long M = *lat.counter;
  const int Q = lat.Kp / 4;
  const long long total = M * Q;
  const int nthreads = gridDim.x * blockDim.x, t0 = blockIdx.x * blockDim.x + threadIdx.x;
  const int2* nbr = lat.nbr + (size_t)j * lat.nc;
  for (long long t = t0; t < total; t += (long long)kBlurIlp * nthreads) {
    size_t self[kBlurIlp], n1[kBlurIlp], n2[kBlurIlp];
    bool ok[kBlurIlp];
#pragma unroll
    for (int u = 0; u < kBlurIlp; ++u) {
      const long long tt = t + (long long)u * nthreads;
      ok[u] = tt < total;
      const int v = ok[u] ? (int)(tt / Q) : 0, q = ok[u] ? (int)(tt - (long long)v * Q) : 0;
      const int2 nb = __ldg(nbr + v);
      self[u] = (size_t)(v + 1) * lat.Kp + 4 * q;
      n1[u] = (size_t)nb.x * lat.Kp + 4 * q;
      n2[u] = (size_t)nb.y * lat.Kp + 4 * q;
    }
    float4 a[kBlurIlp], b[kBlurIlp], c[kBlurIlp];
#pragma unroll
    for (int u = 0; u < kBlurIlp; ++u) {
      a[u] = __ldg(reinterpret_cast<const float4*>(oldv + n1[u]));
      b[u] = __ldg(reinterpret_cast<const float4*>(oldv + n2[u]));
      c[u] = __ldg(reinterpret_cast<const float4*>(oldv + self[u]));
    }
#pragma unroll
    for (int u = 0; u < kBlurIlp; ++u) {
      float4 o;
      o.x = __fadd_rn(c[u].x, __fmul_rn(0.5f, __fadd_rn(a[u].x, b[u].x)));
      o.y = __fadd_rn(c[u].y, __fmul_rn(0.5f, __fadd_rn(a[u].y, b[u].y)));
      o.z = __fadd_rn(c[u].z, __fmul_rn(0.5f, __fadd_rn(a[u].z, b[u].z)));
      o.w = __fadd_rn(c[u].w, __fmul_rn(0.5f, __fadd_rn(a[u].w, b[u].w)));
      if (ok[u]) *reinterpret_cast<float4*>(newv + self[u]) = o;
    }
  }
}

// Slice: out = alpha * sum_r bary_r * values[vertex_r], accumulated in the reference's order.  A group of G lanes (G = 8, 16 or 32
// >= Kp/4) serves one pixel: its six vertex ids / weights are loaded once per lane (broadcast inside the group) and every lane
// gathers 16 bytes of each vertex row, so a row is read with contiguous requests; neighbouring pixels share vertices (L1 hits).
__global__ void __launch_bounds__(256)
lattice_slice_kernel(const float* __restrict__ values_img0, int K, int HW, float alpha, float* __restrict__ out, Lat lat0) {
  extern __shared__ float4 smem4[];   // tile4[Kp/4][kPixTile]
  const Lat lat = for_image(lat0, blockIdx.z);
  const float* values = img_ptr(values_img0, lat.ws, blockIdx.z);
  out += (size_t)blockIdx.z * K * HW;
  const int p0 = blockIdx.x * kPixTile;
  const int Q = lat.Kp / 4;
  const int G = Q <= 8 ? 8 : (Q <= 16 ? 16 : 32), ppw = 32 / G;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q = lane % G, lp = lane / G;
  constexpr int kPixPerWarp = kPixTile / 8;
  for (int qq = q; qq < Q; qq += G) {                  // (one trip: G >= Q = Kp/4 <= 24 for every K <= 96)
    for (int it = 0; it < kPixPerWarp / ppw; ++it) {
      const int p = warp * kPixPerWarp + it * ppw + lp;
      const int pix = p0 + p;
      const float4 s = pix < HW ? slice_quad(lat, values, lat.Kp, pix, qq, alpha) : make_float4(0.f, 0.f, 0.f, 0.f);
      smem4[qq * kPixTile + p] = s;
    }
  }
  __syncthreads();
  const float* tile = reinterpret_cast<const float*>(smem4);
  for (int e = threadIdx.x; e < K * kPixTile; e += blockDim.x) {
    const int k = e / kPixTile, p = e - k * kPixTile;
    if (p0 + p < HW) out[(size_t)k * HW + p0 + p] = tile[((k >> 2) * kPixTile + p) * 4 + (k & 3)];
  }
}

Lat carve_bilateral(void* base, int K, int H, int W) {
  size_t off = 0;
  Lat c = carve<D5, true>(base, &off, (K + 3) / 4 * 4, H, W);
  c.ws = off;
  return c;
}

}  // namespace

// Images are filtered kBatch at a time (grid.z = image); each has its own lattice region in the workspace.
constexpr int kBilateralBatch = 8;

extern "C" size_t acr_bilateral_workspace(int N, int K, int H, int W) {
  if (N <= 0 || K <= 0 || H <= 0 || W <= 0) return 0;
  return carve_bilateral(nullptr, K, H, W).ws * (size_t)(N < kBilateralBatch ? N : kBilateralBatch);
}

extern "C" int acr_bilateral_batch(const float* images, const float* ins, float* outs,
                                   int N, int K, int H, int W, float sigmargb, float sigmaxy,
                                   void* workspace, size_t workspace_bytes, int* lattice_size_host, void* stream) {
  ACR_REQUIRE(images && ins && outs && workspace, ACR_E_INVAL, "acr_bilateral_batch: null pointer");
  ACR_REQUIRE(N > 0 && K > 0 && H > 0 && W > 0, ACR_E_INVAL, "acr_bilateral_batch: bad shape");
  ACR_REQUIRE(sigmargb > 0.f && sigmaxy > 0.f, ACR_E_INVAL, "acr_bilateral_batch: sigma <= 0");
  ACR_REQUIRE((long long)H * W * D6 < (1ll << 28), ACR_E_INVAL, "acr_bilateral_batch: image too large");
  ACR_REQUIRE(((uintptr_t)workspace & 255) == 0, ACR_E_ALIGN, "acr_bilateral_batch: workspace not 256-byte aligned");
  const Lat c = carve_bilateral(workspace, K, H, W);
  ACR_REQUIRE(workspace_bytes >= acr_bilateral_workspace(N, K, H, W), ACR_E_NOMEM, "acr_bilateral_batch: workspace too small (%zu < %zu)",
              workspace_bytes, acr_bilateral_workspace(N, K, H, W));
  cudaStream_t st = (cudaStream_t)stream;
  const int HW = H * W, HWpad = (HW + 3) / 4 * 4, nc = HWpad * D6;

  const Scales<D5> sc = scales<D5>();
  const float alpha = slice_alpha<D5>();

  const size_t smem = (size_t)kPixTile * c.Kp * sizeof(float);      // slice: output tile
  ACR_REQUIRE(smem <= 48 * 1024, ACR_E_INVAL, "acr_bilateral_batch: K=%d too large (<= %d planes)", K, 48 * 1024 / (kPixTile * 4));
  // splat: input tile + four per-pair arrays
  const size_t smem_splat = (size_t)kPixTile * ((c.Kp / 4) | 1) * 16 + (size_t)D6 * kPixTile * 4 * sizeof(int);
  {
    static bool attr_set[64] = {false};
    int dev = 0;
    ACR_CUDA(cudaGetDevice(&dev));
    if (dev >= 0 && dev < 64 && !attr_set[dev]) {
      ACR_CUDA(cudaFuncSetAttribute(lattice_splat_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
      attr_set[dev] = true;
    }
  }
  const int splat_tiles = ((W + kTileW - 1) / kTileW) * ((H + kTileH - 1) / kTileH);
  for (int n0 = 0; n0 < N; n0 += kBilateralBatch) {
    const int nb = (N - n0 < kBilateralBatch) ? N - n0 : kBilateralBatch;
    const float* img = images + (size_t)n0 * 3 * HW;
    const float* in = ins + (size_t)n0 * K * HW;
    float* out = outs + (size_t)n0 * K * HW;
    lattice_embed_kernel<<<dim3((HWpad + 255) / 256, 1, nb), 256, 0, st>>>(img, H, W, sigmargb, sigmaxy, sc, c);
    if (int e = acr::check_launch("lattice_embed_kernel")) return e;
    lattice_insert_kernel<<<dim3((nc + 255) / 256, 1, nb), 256, 0, st>>>(c);
    if (int e = acr::check_launch("lattice_insert_kernel")) return e;
    lattice_prepare_kernel<<<dim3(148 * 4, 1, nb), 256, 0, st>>>(c);
    if (int e = acr::check_launch("lattice_prepare_kernel")) return e;
    lattice_splat_kernel<<<dim3(splat_tiles, 1, nb), 256, smem_splat, st>>>(in, K, H, W, HWpad, c);
    if (int e = acr::check_launch("lattice_splat_kernel")) return e;
    {
      float* cur = c.val0;
      float* nxt = c.val1;
      for (int j = 0; j < D6; ++j) {
        lattice_blur_kernel<<<dim3(148 * 2, 1, nb), 256, 0, st>>>(cur, nxt, j, c);
        if (int e = acr::check_launch("lattice_blur_kernel")) return e;
        float* t = cur; cur = nxt; nxt = t;
      }
    }
    // d+1 = 6 passes (an even number): the result is back in val0
    lattice_slice_kernel<<<dim3((HW + kPixTile - 1) / kPixTile, 1, nb), 256, smem, st>>>(c.val0, K, HW, alpha, out, c);
    if (int e = acr::check_launch("lattice_slice_kernel")) return e;
    if (lattice_size_host) {
      for (int i = 0; i < nb; ++i)
        ACR_CUDA(cudaMemcpyAsync(lattice_size_host + n0 + i, (char*)c.counter + c.ws * i, sizeof(int), cudaMemcpyDeviceToHost, st));
      ACR_CUDA(cudaStreamSynchronize(st));
    }
  }
  return 0;
}

// SWIG-shaped host entry (bilateralfilter.cpp:42-55): HOST buffers in, HOST buffer out.  The device buffers, the lattice workspace
// and the stream are cached per device and only grow (the reference allocates and frees its lattice on every call).
namespace {
struct HostCache {
  float *img = nullptr, *in = nullptr, *out = nullptr;
  void* ws = nullptr;
  size_t img_b = 0, io_b = 0, ws_b = 0;
  cudaStream_t st = nullptr;
};
std::mutex g_host_mutex;
HostCache g_host_cache[64];

cudaError_t grow(void** p, size_t* have, size_t need) {
  if (*have >= need) return cudaSuccess;
  if (*p) cudaFree(*p);
  *p = nullptr;
  *have = 0;
  cudaError_t e = cudaMalloc(p, need);
  if (e == cudaSuccess) *have = need;
  return e;
}
}  // namespace

extern "C" void bilateralfilter_batch_b200(const float* images_host, int len_images, const float* ins_host, int len_ins,
                                           float* outs_host, int len_outs,
                                           int N, int K, int H, int W, float sigmargb, float sigmaxy) {
  const long long hw = (long long)H * W;
  if (!images_host || !ins_host || !outs_host || N <= 0 || K <= 0 || hw <= 0 ||
      (long long)len_images != 3 * hw * N || (long long)len_ins != K * hw * N || len_outs != len_ins) {
    acr::set_error("bilateralfilter_batch_b200: buffer lengths do not match N=%d K=%d H=%d W=%d", N, K, H, W);
    return;
  }
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess || dev < 0 || dev >= 64) { acr::set_error("bilateralfilter_batch_b200: cudaGetDevice: %s", cudaGetErrorString(e)); return; }
  std::lock_guard<std::mutex> lock(g_host_mutex);
  HostCache& hc = g_host_cache[dev];
  auto fail = [&](const char* what) { acr::set_error("bilateralfilter_batch_b200: %s: %s", what, cudaGetErrorString(e)); };
  if (!hc.st && (e = cudaStreamCreateWithFlags(&hc.st, cudaStreamNonBlocking)) != cudaSuccess) { hc.st = nullptr; return fail("cudaStreamCreate"); }
  const size_t ws_bytes = acr_bilateral_workspace(N, K, H, W);
  size_t in_b = hc.io_b, out_b = hc.io_b;
  if ((e = grow((void**)&hc.img, &hc.img_b, (size_t)len_images * 4)) != cudaSuccess) return fail("cudaMalloc(images)");
  if ((e = grow((void**)&hc.in, &in_b, (size_t)len_ins * 4)) != cudaSuccess) { hc.io_b = 0; return fail("cudaMalloc(ins)"); }
  if ((e = grow((void**)&hc.out, &out_b, (size_t)len_outs * 4)) != cudaSuccess) { hc.io_b = 0; return fail("cudaMalloc(outs)"); }
  hc.io_b = in_b < out_b ? in_b : out_b;
  if ((e = grow(&hc.ws, &hc.ws_b, ws_bytes)) != cudaSuccess) return fail("cudaMalloc(workspace)");
  if ((e = cudaMemcpyAsync(hc.img, images_host, (size_t)len_images * 4, cudaMemcpyHostToDevice, hc.st)) != cudaSuccess) return fail("H2D images");
  if ((e = cudaMemcpyAsync(hc.in, ins_host, (size_t)len_ins * 4, cudaMemcpyHostToDevice, hc.st)) != cudaSuccess) return fail("H2D ins");
  if (acr_bilateral_batch(hc.img, hc.in, hc.out, N, K, H, W, sigmargb, sigmaxy, hc.ws, hc.ws_b, nullptr, hc.st) != 0) return;   // error string already set
  if ((e = cudaMemcpyAsync(outs_host, hc.out, (size_t)len_outs * 4, cudaMemcpyDeviceToHost, hc.st)) != cudaSuccess) return fail("D2H outs");
  if ((e = cudaStreamSynchronize(hc.st)) != cudaSuccess) return fail("synchronize");
  acr::set_error("");
}
