// Dense-CRF mean-field inference on the GPU: densecrf 2.x (the library under pydensecrf) as the PSA-lineage
// crf_inference(img, probs, t, scale_factor, labels) of tool/imutils.py:345-399 drives it.
//
// Per image (C labels, HW pixels):
//   -U      = log(max(P, clip))                                      (unary_from_softmax; P need not sum to 1)
//   Q0      = softmax_c(-U)                                          (expAndNormalize: max subtracted, exp, divided by the sum)
//   K_k(v)  = norm_k * L_k(norm_k * v),  norm_k = 1 / sqrt(L_k(1) + 1e-20)      (DIAG_KERNEL, NORMALIZE_SYMMETRIC)
//   Q      <- softmax_c(-U + compat_g * K_g(Q) + compat_b * K_b(Q))  n_iter times (Potts: compatibility -w*Q, subtracted)
// L_g is the permutohedral filter over (x/sxy_g, y/sxy_g) (d = 2), L_b over (x/sxy_b, y/sxy_b, r/srgb, g/srgb, b/srgb)
// (d = 5), both with densecrf 2.x's scalar embedding (lattice.cuh, Pad = false).
//
// Launches per batch of up to 8 images (grid.z = image, grid.y = lattice): 11 + 8 * n_iter.
//   embed, insert, prepare     both lattices of every image, once
//   normalisation pass         splat of a plane of ones, d+1 = 6 blur passes (the Gaussian lattice takes part in the first
//                              3), then `update` in its first mode: norm_g, norm_b and Q0
//   per iteration              splat (norm * Q folded into the splat's tile load; Q is never rewritten), 6 blur passes,
//                              `update`: both slices, -U + both terms, softmax over the planes, Q written in place
//
// Determinism.  The splat adds the (pixel, vertex) contributions of a vertex in whatever order its CTAs finish, so it adds them
// as 64-bit fixed point (scale 2^32) with integer reduce-adds, whose sum does not depend on the order; two calls, and an image
// run alone or inside a batch, give the same bits.  The first blur pass converts to fp32, the last one zeroes the accumulators.
// Range: bary in [0,1], Q in [0,1] and norm <= 1/sqrt(alpha/(d+1)) (L(1) at a pixel is at least alpha * sum_r bary_r^2 >=
// alpha/(d+1): the blur only adds non-negative terms to the pixel's own splat) = 2.49 for d = 5, 1.94 for d = 2.  So one
// contribution is below 4 = 2^34 in fixed point, and a vertex receives at most (d+1)*HW < 2^28 of them (checked on entry):
// |sum| < 2^62 never wraps.  A contribution outside [-4, 4] (or NaN, from non-finite scores) sets the image's flag, and the
// softmax then writes NaN for every Q of that image instead of a silently wrapped result.
#include "lattice.cuh"
#include <cmath>

namespace {

using namespace acr::lattice;
using LatG = Lattice<2>;
using LatB = Lattice<5>;

constexpr int kBatch = 8;           // images per launch (grid.z)
constexpr int kMaxC = 96;           // update tile: 128 pixels x 96 planes x 4 B = 48 KB of shared memory
constexpr int kPixTile = 128;       // pixels per CTA (splat: 16 x 8 block of the image; update: 128 consecutive pixels)
constexpr int kTileW = 16, kTileH = 8;
constexpr int kSlotProbes = 32;
constexpr int kSplatSlots = 1024;   // >= the 768 pairs of a tile, so the table never fills up; 4 slots per thread in the scan
constexpr int kBlurIlp = 4;
constexpr float kFix = 4294967296.f;          // fixed-point scale 2^32
constexpr float kPairMax = 4.f;               // largest |contribution| (see the range argument above)

struct Crf {
  LatG g;
  LatB b;
  long long *acc_g, *acc_b;     // fixed-point splat accumulators [(nc+1) * Kp]; all zero between passes
  float *norm_g, *norm_b;       // [HW]
  int* flag;                    // != 0: a splat contribution left the fixed-point range
  size_t ws;
};

__device__ __forceinline__ Crf for_image(const Crf& c, int n) {
  Crf r = c;
  r.g = for_image(c.g, n);
  r.b = for_image(c.b, n);
  r.acc_g = img_ptr(c.acc_g, c.ws, n); r.acc_b = img_ptr(c.acc_b, c.ws, n);
  r.norm_g = img_ptr(c.norm_g, c.ws, n); r.norm_b = img_ptr(c.norm_b, c.ws, n);
  r.flag = img_ptr(c.flag, c.ws, n);
  return r;
}

__global__ void __launch_bounds__(256)
crf_embed_kernel(const float* __restrict__ images, int H, int W, float sxy_g, float sxy_b, float srgb, Scales<2> sc_g,
                 Scales<5> sc_b, Crf c0) {
  const Crf c = for_image(c0, blockIdx.z);
  const int idx = blockIdx.x * blockDim.x + threadIdx.x, gthreads = gridDim.x * blockDim.x;
  if (blockIdx.y == 0) {
    embed<2, false>(c.g, nullptr, H, W, srgb, sxy_g, sc_g, idx, gthreads);
    if (idx == 0) *c.flag = 0;
  } else {
    embed<5, false>(c.b, images + (size_t)blockIdx.z * 3 * H * W, H, W, srgb, sxy_b, sc_b, idx, gthreads);
  }
}

__global__ void __launch_bounds__(256)
crf_insert_kernel(Crf c0) {
  const Crf c = for_image(c0, blockIdx.z);
  const int cand = blockIdx.x * blockDim.x + threadIdx.x;
  if (blockIdx.y == 0) {
    if ((int)(blockIdx.x * blockDim.x) < c.g.nc) insert(c.g, cand);        // the Gaussian lattice has half the candidates
  } else {
    insert(c.b, cand);
  }
}

// Blur neighbours, candidate -> vertex, zeroed accumulators and slot 0 (the missing neighbour) of both value arrays.
template <int D>
__device__ __forceinline__ void prepare_lattice(const Lattice<D>& lat, long long* acc, int t0, int nthreads) {
  prepare(lat, t0, nthreads);
  const long long nz = ((long long)*lat.counter + 1) * lat.Kp / 2;
  longlong2* z = reinterpret_cast<longlong2*>(acc);
  for (long long i = t0; i < nz; i += nthreads) z[i] = make_longlong2(0, 0);
  if (t0 < lat.Kp) { lat.val0[t0] = 0.f; lat.val1[t0] = 0.f; }
}

__global__ void __launch_bounds__(256)
crf_prepare_kernel(Crf c0) {
  const Crf c = for_image(c0, blockIdx.z);
  const int nthreads = gridDim.x * blockDim.x, t0 = blockIdx.x * blockDim.x + threadIdx.x;
  if (blockIdx.y == 0) prepare_lattice(c.g, c.acc_g, t0, nthreads);
  else prepare_lattice(c.b, c.acc_b, t0, nthreads);
}

__device__ __forceinline__ long long to_fixed(float v, bool& bad) {
  bad |= !(fabsf(v) <= kPairMax);
  return __float2ll_rn(v * kFix);
}
__device__ __forceinline__ void red_add_s64(long long* addr, long long v) {
  atomicAdd(reinterpret_cast<unsigned long long*>(addr), (unsigned long long)v);
}

struct SplatShared {
  int skey[kSplatSlots], scount[kSplatSlots], sstart[kSplatSlots], socc[kSplatSlots], warp_tot[8], warp_occ[8], n_occ;
};

// Splat of one 16 x 8 pixel block into one lattice.  Same shape as the bilateral filter's splat (lattice_splat_kernel): the
// (pixel, remainder) pairs are sorted by vertex in shared memory with integer atomics, then one work item per (vertex, 4 planes)
// sums its pairs and issues one reduce-add per plane -- here in fixed point.
// q == nullptr: the normalisation pass (one plane of ones); otherwise planes norm * q[k] for k < C, nq = Kp/4 quads.
template <int D>
__device__ __forceinline__ void splat_tile(const Lattice<D>& lat, long long* __restrict__ acc, const float* __restrict__ norm,
                                           const float* __restrict__ q, int C, int H, int W, int nq, int* flag, SplatShared& sh,
                                           float4* smem4) {
  constexpr int NP = (D + 1) * kPixTile;
  const int HW = H * W, Kp = lat.Kp;
  const int Qs = nq | 1;                                // odd row stride (in float4): conflict-free 128-bit stores
  int* slot = reinterpret_cast<int*>(smem4 + (size_t)Qs * kPixTile);      // [NP]: slot of the pair, -1 = none
  int* pos = slot + NP;                                                   // position inside the slot
  int* order = pos + NP;                                                  // pair indices sorted by slot
  float* wts = reinterpret_cast<float*>(order + NP);
  const int tiles_x = (W + kTileW - 1) / kTileW;
  const int x0 = (blockIdx.x % tiles_x) * kTileW, y0 = (blockIdx.x / tiles_x) * kTileH;
  bool bad = false;
  for (int i = threadIdx.x; i < kSplatSlots; i += blockDim.x) { sh.skey[i] = 0; sh.scount[i] = 0; }
  for (int e = threadIdx.x; e < nq * kPixTile; e += blockDim.x) {
    const int qd = e / kPixTile, p = e - qd * kPixTile;
    const int x = x0 + (p % kTileW), y = y0 + (p / kTileW);
    const bool in = x < W && y < H;
    const size_t pix = (size_t)y * W + x;
    const float nrm = (q && in) ? __ldg(norm + pix) : 1.f;
    float v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = 4 * qd + j;
      v[j] = (k < C && in) ? (q ? __fmul_rn(nrm, __ldg(q + (size_t)k * HW + pix)) : 1.f) : 0.f;
    }
    smem4[p * Qs + qd] = make_float4(v[0], v[1], v[2], v[3]);
  }
  __syncthreads();
  for (int w = threadIdx.x; w < NP; w += blockDim.x) {
    const int p = w % kPixTile, r = w / kPixTile;
    const int x = x0 + (p % kTileW), y = y0 + (p / kTileW);
    int sl = -1;
    float wt = 0.f;
    if (x < W && y < H) {
      const int pix = y * W + x;
      const int o = __ldg(lat.offs + (size_t)r * lat.hwp + pix);
      wt = __ldg(lat.bary + (size_t)r * lat.hwp + pix);
      const uint32_t h = ((uint32_t)o * 0x9E3779B1u) >> 7;
      for (int t = 0; t < kSlotProbes; ++t) {
        const int i = (int)((h + t) & (uint32_t)(kSplatSlots - 1));
        const int prev = atomicCAS(&sh.skey[i], 0, o);
        if (prev == 0 || prev == o) { sl = i; break; }
      }
      if (sl >= 0) {
        pos[w] = atomicAdd(&sh.scount[sl], 1);
      } else {                                          // table neighbourhood full (rare): this pair adds to global memory itself
        for (int qd = 0; qd < nq; ++qd) {
          const float4 xv = smem4[p * Qs + qd];
          const float c4[4] = {xv.x, xv.y, xv.z, xv.w};
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (4 * qd + j < C) red_add_s64(acc + (size_t)o * Kp + 4 * qd + j, to_fixed(__fmul_rn(wt, c4[j]), bad));
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
    int cnt[PER], tot = 0, occ = 0;
#pragma unroll
    for (int u = 0; u < PER; ++u) { cnt[u] = sh.scount[threadIdx.x * PER + u]; tot += cnt[u]; occ += cnt[u] > 0; }
    int v = tot, vo = occ;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int n = __shfl_up_sync(0xffffffffu, v, o), no = __shfl_up_sync(0xffffffffu, vo, o);
      if (lane >= o) { v += n; vo += no; }
    }
    if (lane == 31) { sh.warp_tot[wp] = v; sh.warp_occ[wp] = vo; }
    __syncthreads();
    int base = v - tot, obase = vo - occ;
    for (int i = 0; i < wp; ++i) { base += sh.warp_tot[i]; obase += sh.warp_occ[i]; }
#pragma unroll
    for (int u = 0; u < PER; ++u) {
      sh.sstart[threadIdx.x * PER + u] = base;
      base += cnt[u];
      if (cnt[u] > 0) sh.socc[obase++] = threadIdx.x * PER + u;
    }
    if (threadIdx.x == blockDim.x - 1) sh.n_occ = obase;
  }
  __syncthreads();
  for (int w = threadIdx.x; w < NP; w += blockDim.x) {
    const int sl = slot[w];
    if (sl >= 0) order[sh.sstart[sl] + pos[w]] = w;
  }
  __syncthreads();
  const int nitems = sh.n_occ * nq;
  for (int w = threadIdx.x; w < nitems; w += blockDim.x) {
    const int sidx = sh.socc[w / nq], qd = w % nq;
    const int beg = sh.sstart[sidx], n = sh.scount[sidx];
    long long a0 = 0, a1 = 0, a2 = 0, a3 = 0;
    for (int j = 0; j < n; ++j) {
      const int pw = order[beg + j];
      const float wt = wts[pw];
      const float4 xv = smem4[(pw % kPixTile) * Qs + qd];
      a0 += to_fixed(__fmul_rn(wt, xv.x), bad);
      a1 += to_fixed(__fmul_rn(wt, xv.y), bad);
      a2 += to_fixed(__fmul_rn(wt, xv.z), bad);
      a3 += to_fixed(__fmul_rn(wt, xv.w), bad);
    }
    long long* dst = acc + (size_t)sh.skey[sidx] * Kp + 4 * qd;
    const int k0 = 4 * qd;
    red_add_s64(dst, a0);
    if (k0 + 1 < C) red_add_s64(dst + 1, a1);
    if (k0 + 2 < C) red_add_s64(dst + 2, a2);
    if (k0 + 3 < C) red_add_s64(dst + 3, a3);
  }
  if (bad) atomicExch(flag, 1);
}

__global__ void __launch_bounds__(256)
crf_splat_kernel(const float* __restrict__ q, int C, int H, int W, int nq, Crf c0) {
  extern __shared__ float4 smem4[];                    // tile4[kPixTile][nq | 1], then the per-pair arrays
  __shared__ SplatShared sh;
  const Crf c = for_image(c0, blockIdx.z);
  if (q) q += (size_t)blockIdx.z * C * H * W;
  if (blockIdx.y == 0) splat_tile(c.g, c.acc_g, c.norm_g, q, C, H, W, nq, c.flag, sh, smem4);
  else splat_tile(c.b, c.acc_b, c.norm_b, q, C, H, W, nq, c.flag, sh, smem4);
}

// Blur pass j of one lattice: new = old + 0.5 * (old[n1] + old[n2]), items (vertex, 4 planes) of the first nq quads of each row.
// Pass 0 reads the fixed-point accumulators into val0, pass j >= 1 goes val0 -> val1 (j odd) or val1 -> val0 (j even), so
// the result of the d+1 passes is in val0 for d = 2 and in val1 for d = 5.  The last pass zeroes the accumulators.
__device__ __forceinline__ float4 load_vals(const long long* acc, size_t i) {
  const longlong2 a = __ldg(reinterpret_cast<const longlong2*>(acc + i)), b = __ldg(reinterpret_cast<const longlong2*>(acc + i + 2));
  const float s = 1.f / kFix;
  return make_float4(__ll2float_rn(a.x) * s, __ll2float_rn(a.y) * s, __ll2float_rn(b.x) * s, __ll2float_rn(b.y) * s);
}
__device__ __forceinline__ float4 load_vals(const float* v, size_t i) { return __ldg(reinterpret_cast<const float4*>(v + i)); }

template <int D, typename Src>
__device__ __forceinline__ void blur_pass(const Lattice<D>& lat, const Src* __restrict__ src, float* __restrict__ dst, int j, int nq,
                                          int t0, int nthreads) {
  const long long total = (long long)*lat.counter * nq;
  const int Kp = lat.Kp;
  const int2* nbr = lat.nbr + (size_t)j * lat.nc;
  for (long long t = t0; t < total; t += (long long)kBlurIlp * nthreads) {
    size_t self[kBlurIlp], n1[kBlurIlp], n2[kBlurIlp];
    bool ok[kBlurIlp];
#pragma unroll
    for (int u = 0; u < kBlurIlp; ++u) {
      const long long tt = t + (long long)u * nthreads;
      ok[u] = tt < total;
      const int v = ok[u] ? (int)(tt / nq) : 0, qd = ok[u] ? (int)(tt - (long long)v * nq) : 0;
      const int2 nb = __ldg(nbr + v);
      self[u] = (size_t)(v + 1) * Kp + 4 * qd;
      n1[u] = (size_t)nb.x * Kp + 4 * qd;
      n2[u] = (size_t)nb.y * Kp + 4 * qd;
    }
    float4 a[kBlurIlp], b[kBlurIlp], c[kBlurIlp];
#pragma unroll
    for (int u = 0; u < kBlurIlp; ++u) {
      a[u] = load_vals(src, n1[u]);
      b[u] = load_vals(src, n2[u]);
      c[u] = load_vals(src, self[u]);
    }
#pragma unroll
    for (int u = 0; u < kBlurIlp; ++u) {
      float4 o;
      o.x = __fadd_rn(c[u].x, __fmul_rn(0.5f, __fadd_rn(a[u].x, b[u].x)));
      o.y = __fadd_rn(c[u].y, __fmul_rn(0.5f, __fadd_rn(a[u].y, b[u].y)));
      o.z = __fadd_rn(c[u].z, __fmul_rn(0.5f, __fadd_rn(a[u].z, b[u].z)));
      o.w = __fadd_rn(c[u].w, __fmul_rn(0.5f, __fadd_rn(a[u].w, b[u].w)));
      if (ok[u]) *reinterpret_cast<float4*>(dst + self[u]) = o;
    }
  }
}

template <int D>
__device__ __forceinline__ void blur_lattice(const Lattice<D>& lat, long long* acc, int j, int nq, int t0, int nthreads) {
  if (j == 0) blur_pass(lat, acc, lat.val0, j, nq, t0, nthreads);
  else if (j & 1) blur_pass(lat, lat.val0, lat.val1, j, nq, t0, nthreads);
  else blur_pass(lat, lat.val1, lat.val0, j, nq, t0, nthreads);
  if (j == D) {
    const long long total = (long long)*lat.counter * nq;
    for (long long t = t0; t < total; t += nthreads) {
      const int v = (int)(t / nq), qd = (int)(t - (long long)v * nq);
      longlong2* z = reinterpret_cast<longlong2*>(acc + (size_t)(v + 1) * lat.Kp + 4 * qd);
      z[0] = make_longlong2(0, 0);
      z[1] = make_longlong2(0, 0);
    }
  }
}

// grid.y = 2 for passes 0..2 (y = 1: the Gaussian lattice), 1 for passes 3..5.
__global__ void __launch_bounds__(256)
crf_blur_kernel(int j, int nq, Crf c0) {
  const Crf c = for_image(c0, blockIdx.z);
  const int nthreads = gridDim.x * blockDim.x, t0 = blockIdx.x * blockDim.x + threadIdx.x;
  if (blockIdx.y == 0) blur_lattice(c.b, c.acc_b, j, nq, t0, nthreads);
  else blur_lattice(c.g, c.acc_g, j, nq, t0, nthreads);
}

// 128 consecutive pixels of one image, all planes in shared memory (tile4[Kp/4][128]):
//   1. -U = log(max(P, clip)) for every plane;
//   2. init: norm_k = 1/sqrt(L_k(1) + 1e-20) from plane 0 of the normalisation pass (in double, as densecrf 2.x), logits = -U;
//      otherwise: logits = -U + compat_g * (norm_g * S_g) + compat_b * (norm_b * S_b), S_k the slices of the blurred lattices;
//   3. softmax over the C planes per pixel (max subtracted, exp, divided by the sum), Q written (NaN if the image's flag is set).
__global__ void __launch_bounds__(256)
crf_update_kernel(const float* __restrict__ P, float* __restrict__ Q, int C, int HW, float clip, float compat_g, float compat_b,
                  float alpha_g, float alpha_b, int init, Crf c0) {
  extern __shared__ float4 tile4[];
  float* tile = reinterpret_cast<float*>(tile4);
  const Crf c = for_image(c0, blockIdx.z);
  P += (size_t)blockIdx.z * C * HW;
  Q += (size_t)blockIdx.z * C * HW;
  const int p0 = blockIdx.x * kPixTile;
  const int Kp = c.b.Kp, nq = Kp / 4;
  for (int e = threadIdx.x; e < C * kPixTile; e += blockDim.x) {
    const int k = e / kPixTile, p = e - k * kPixTile;
    tile[((k >> 2) * kPixTile + p) * 4 + (k & 3)] = p0 + p < HW ? logf(fmaxf(__ldg(P + (size_t)k * HW + p0 + p), clip)) : 0.f;
  }
  if (init) {
    const int pix = p0 + threadIdx.x;
    if (threadIdx.x < kPixTile && pix < HW) {
      const float sg = slice_quad(c.g, c.g.val0, Kp, pix, 0, alpha_g).x;
      const float sb = slice_quad(c.b, c.b.val1, Kp, pix, 0, alpha_b).x;
      c.norm_g[pix] = (float)__ddiv_rn(1.0, __dsqrt_rn(__dadd_rn((double)sg, 1e-20)));
      c.norm_b[pix] = (float)__ddiv_rn(1.0, __dsqrt_rn(__dadd_rn((double)sb, 1e-20)));
    }
    __syncthreads();
  } else {
    __syncthreads();
    // a group of G lanes (G >= nq) serves one pixel; every lane gathers 16 bytes of each vertex row
    const int G = nq <= 8 ? 8 : (nq <= 16 ? 16 : 32), ppw = 32 / G;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int qq = lane % G, lp = lane / G;
    constexpr int kPixPerWarp = kPixTile / 8;
    if (qq < nq) {
      for (int it = 0; it < kPixPerWarp / ppw; ++it) {
        const int p = warp * kPixPerWarp + it * ppw + lp;
        const int pix = p0 + p;
        if (pix >= HW) continue;
        const float4 sg = slice_quad(c.g, c.g.val0, Kp, pix, qq, alpha_g);
        const float4 sb = slice_quad(c.b, c.b.val1, Kp, pix, qq, alpha_b);
        const float ng = __ldg(c.norm_g + pix), nb = __ldg(c.norm_b + pix);
        float4 t = tile4[qq * kPixTile + p];
        t.x = __fadd_rn(__fadd_rn(t.x, __fmul_rn(compat_g, __fmul_rn(ng, sg.x))), __fmul_rn(compat_b, __fmul_rn(nb, sb.x)));
        t.y = __fadd_rn(__fadd_rn(t.y, __fmul_rn(compat_g, __fmul_rn(ng, sg.y))), __fmul_rn(compat_b, __fmul_rn(nb, sb.y)));
        t.z = __fadd_rn(__fadd_rn(t.z, __fmul_rn(compat_g, __fmul_rn(ng, sg.z))), __fmul_rn(compat_b, __fmul_rn(nb, sb.z)));
        t.w = __fadd_rn(__fadd_rn(t.w, __fmul_rn(compat_g, __fmul_rn(ng, sg.w))), __fmul_rn(compat_b, __fmul_rn(nb, sb.w)));
        tile4[qq * kPixTile + p] = t;
      }
    }
    __syncthreads();
  }
  const int p = threadIdx.x, pix = p0 + p;
  if (p >= kPixTile || pix >= HW) return;
  const bool bad = *c.flag != 0;
  auto at = [&](int k) -> float& { return tile[((k >> 2) * kPixTile + p) * 4 + (k & 3)]; };
  float m = -INFINITY;
  for (int k = 0; k < C; ++k) m = fmaxf(m, at(k));
  float s = 0.f;
  for (int k = 0; k < C; ++k) {
    const float e = expf(__fsub_rn(at(k), m));
    at(k) = e;
    s = __fadd_rn(s, e);
  }
  for (int k = 0; k < C; ++k) Q[(size_t)k * HW + pix] = bad ? __int_as_float(0x7fc00000) : __fdiv_rn(at(k), s);
}

Crf carve_crf(void* base, int C, int H, int W) {
  const int Kp = (C + 3) / 4 * 4;
  size_t off = 0;
  Crf c{};
  c.g = carve<2, false>(base, &off, Kp, H, W);
  c.b = carve<5, false>(base, &off, Kp, H, W);
  auto take = [&](size_t bytes) { size_t o = off; off += acr::align_up(bytes, 256); return (char*)base + o; };
  c.acc_g = (long long*)take(((size_t)c.g.nc + 1) * Kp * sizeof(long long));
  c.acc_b = (long long*)take(((size_t)c.b.nc + 1) * Kp * sizeof(long long));
  c.norm_g = (float*)take((size_t)H * W * sizeof(float));
  c.norm_b = (float*)take((size_t)H * W * sizeof(float));
  c.flag = (int*)take(sizeof(int));
  c.ws = c.g.ws = c.b.ws = off;
  return c;
}

bool positive_finite(float v) { return std::isfinite(v) && v > 0.f; }

// Largest |key coordinate| the embedding can produce for features up to fmax (elevated[j] is a sum of terms (i+1)*scale_i*f_i
// at most; the remainder-0 point, the wrap-around, the canonical offset and the blur neighbours add < 4(d+1)).
template <int D> double key_bound(const float* fmax) {
  const Scales<D> sc = scales<D>();
  double b = 0.0;
  for (int i = 0; i < D; ++i) b += (i + 1) * (double)sc.s[i] * fmax[i];
  return b + 4.0 * (D + 1);
}

}  // namespace

extern "C" size_t acr_dense_crf_workspace(int N, int C, int H, int W) {
  if (N <= 0 || C <= 0 || C > kMaxC || H <= 0 || W <= 0 || (long long)H * W * 6 >= (1ll << 28)) return 0;
  return carve_crf(nullptr, C, H, W).ws * (size_t)(N < kBatch ? N : kBatch);
}

extern "C" int acr_dense_crf(const float* images, const float* probs, float* q_out, int N, int C, int H, int W, int n_iter,
                             float sxy_g, float compat_g, float sxy_b, float srgb, float compat_b, float clip,
                             void* ws, size_t ws_bytes, void* stream) {
  ACR_REQUIRE(images && probs && q_out && ws, ACR_E_INVAL, "acr_dense_crf: null pointer");
  ACR_REQUIRE(N > 0 && C > 0 && H > 0 && W > 0, ACR_E_INVAL, "acr_dense_crf: bad shape N=%d C=%d H=%d W=%d", N, C, H, W);
  ACR_REQUIRE(C <= kMaxC, ACR_E_INVAL, "acr_dense_crf: C=%d > %d labels", C, kMaxC);
  ACR_REQUIRE((long long)H * W * 6 < (1ll << 28), ACR_E_INVAL, "acr_dense_crf: image too large (6*H*W >= 2^28)");
  ACR_REQUIRE(n_iter >= 0, ACR_E_INVAL, "acr_dense_crf: n_iter < 0");
  ACR_REQUIRE(positive_finite(sxy_g) && positive_finite(sxy_b) && positive_finite(srgb), ACR_E_INVAL,
              "acr_dense_crf: sigmas must be finite and > 0");
  ACR_REQUIRE(std::isfinite(compat_g) && std::isfinite(compat_b), ACR_E_INVAL, "acr_dense_crf: compat not finite");
  ACR_REQUIRE(clip > 0.f && clip <= 1.f, ACR_E_INVAL, "acr_dense_crf: clip outside (0, 1]");
  {   // keys are int16: the spatial extent over sxy (and 255/srgb for 0..255 colours) must keep them in range
    const float fg[2] = {(W - 1) / sxy_g, (H - 1) / sxy_g};
    const float fb[5] = {(W - 1) / sxy_b, (H - 1) / sxy_b, 255.f / srgb, 255.f / srgb, 255.f / srgb};
    ACR_REQUIRE(key_bound<2>(fg) <= 32767.0 && key_bound<5>(fb) <= 32767.0, ACR_E_INVAL,
                "acr_dense_crf: lattice coordinates overflow int16 (sigmas too small for a %dx%d image)", H, W);
  }
  ACR_REQUIRE(((uintptr_t)ws & 255) == 0, ACR_E_ALIGN, "acr_dense_crf: workspace not 256-byte aligned");
  const size_t need = acr_dense_crf_workspace(N, C, H, W);
  ACR_REQUIRE(ws_bytes >= need, ACR_E_NOMEM, "acr_dense_crf: workspace too small (%zu < %zu)", ws_bytes, need);

  cudaStream_t st = (cudaStream_t)stream;
  const Crf c = carve_crf(ws, C, H, W);
  const int HW = H * W, nq = c.b.Kp / 4;
  const Scales<2> sc_g = scales<2>();
  const Scales<5> sc_b = scales<5>();
  const float alpha_g = slice_alpha<2>(), alpha_b = slice_alpha<5>();
  const size_t smem_update = (size_t)kPixTile * c.b.Kp * sizeof(float);
  auto smem_splat = [](int q) { return (size_t)kPixTile * (q | 1) * 16 + (size_t)6 * kPixTile * 4 * sizeof(int); };
  {
    static bool attr_set[64] = {false};
    int dev = 0;
    ACR_CUDA(cudaGetDevice(&dev));
    if (dev >= 0 && dev < 64 && !attr_set[dev]) {
      ACR_CUDA(cudaFuncSetAttribute(crf_splat_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_splat(kMaxC / 4)));
      attr_set[dev] = true;
    }
  }
  const int splat_tiles = ((W + kTileW - 1) / kTileW) * ((H + kTileH - 1) / kTileH);
  const int update_tiles = (HW + kPixTile - 1) / kPixTile;
  for (int n0 = 0; n0 < N; n0 += kBatch) {
    const int nb = (N - n0 < kBatch) ? N - n0 : kBatch;
    const float* img = images + (size_t)n0 * 3 * HW;
    const float* P = probs + (size_t)n0 * C * HW;
    float* Q = q_out + (size_t)n0 * C * HW;
    crf_embed_kernel<<<dim3((HW + 255) / 256, 2, nb), 256, 0, st>>>(img, H, W, sxy_g, sxy_b, srgb, sc_g, sc_b, c);
    if (int e = acr::check_launch("crf_embed_kernel")) return e;
    crf_insert_kernel<<<dim3((c.b.nc + 255) / 256, 2, nb), 256, 0, st>>>(c);
    if (int e = acr::check_launch("crf_insert_kernel")) return e;
    crf_prepare_kernel<<<dim3(148 * 4, 2, nb), 256, 0, st>>>(c);
    if (int e = acr::check_launch("crf_prepare_kernel")) return e;
    // pass -1: the normalisation (a plane of ones, one quad); then n_iter mean-field iterations
    for (int it = -1; it < n_iter; ++it) {
      const bool init = it < 0;
      const int q = init ? 1 : nq;
      crf_splat_kernel<<<dim3(splat_tiles, 2, nb), 256, smem_splat(q), st>>>(init ? nullptr : Q, init ? 1 : C, H, W, q, c);
      if (int e = acr::check_launch("crf_splat_kernel")) return e;
      for (int j = 0; j < 6; ++j) {
        crf_blur_kernel<<<dim3(148 * 2, j <= 2 ? 2 : 1, nb), 256, 0, st>>>(j, q, c);
        if (int e = acr::check_launch("crf_blur_kernel")) return e;
      }
      crf_update_kernel<<<dim3(update_tiles, 1, nb), 256, smem_update, st>>>(P, Q, C, HW, clip, compat_g, compat_b, alpha_g,
                                                                              alpha_b, init ? 1 : 0, c);
      if (int e = acr::check_launch("crf_update_kernel")) return e;
    }
  }
  return 0;
}
