// Pseudo-label evaluation (evaluation.py:28-67): the per-class P / T / TP counts of label_iou, for the argmax pseudo-label of
// pseudo_label at EVERY background threshold of a sweep in one pass over the CAMs.
//
// At a pixel whose first maximum over the classes is c* with value m, the pseudo-label at threshold tau is c* when
// m > float32(tau) and background otherwise.  So a pixel only needs j = #{thresholds < m}: it is labelled c* at thresholds
// 0..j-1 and background at j..T-1.  The kernel histograms (c*, j), (c* == gt, j), (gt == 0, j) and gt; prefix / suffix sums
// of these (torch int64 on the device, cam.py) give P, T and TP at every threshold exactly.
//
// Work: tiles of kTile pixels of one image; a CTA takes a contiguous range of tiles, counts into shared-memory u32
// histograms (warp-aggregated with __match_any_sync: most pixels of a warp share a bin) and flushes the non-zero bins into
// the caller's int64 counters with integer atomics.  Integer sums do not depend on their order: the counts are bitwise
// deterministic, and they accumulate across calls.
#include "attn_tc.cuh"      // acr_attn::set_max_smem
#include <algorithm>
#include <cmath>
#include <cstring>
#include <vector>

namespace {

constexpr int kThreads = 256;
constexpr int kPer = 8;                                // pixels per thread and tile
constexpr int kTile = kThreads * kPer;                 // pixels per tile
// No u32 counter can overflow: a pixel adds 1 to at most one bin of each histogram, and a CTA counts at most
// kMaxTilesPerCta * kTile = 2^31 pixels before it flushes; the int64 device counters take the sums across CTAs and calls.
constexpr long long kMaxTilesPerCta = 1LL << 20;
constexpr int kMaxThresholds = 4096;
constexpr size_t kMaxHist = 200 * 1024;               // (2K-1)(T+1)*4 + 4K, as cam_finish's cap
constexpr size_t kMaxSmem = kMaxHist + 4 + kMaxThresholds * sizeof(float);    // + the bin of gt >= K, + the thresholds

// Device copy of the host tables (one cudaMemcpyAsync per call).  Per image: offset of its ground truth (and, in label-map
// mode, of its prediction), pixel count, first tile, and its planes sorted by class with the first class that has no plane
// (an implicit zero plane; K when every class has one) and the first candidate class (= min of both).
struct Img {
  long long off, npix, tile0, plane0, nplanes, zero_label, first_label, pad;
};
struct Plane {
  long long off, label;                                // label = dict class + 1
};

struct CamParams {
  const float* cams;
  const unsigned char* gt;
  unsigned long long* counts;
  const Img* img;
  const Plane* planes;
  const float* thr;
  int num_images, K, T;
  long long total_tiles, tiles_per_cta;
};

struct MapParams {
  const unsigned char* pred;
  const unsigned char* gt;
  unsigned long long* counts;
  const Img* img;
  int num_images, K;
  long long total_tiles, tiles_per_cta;
};

// Calls f(image row, first pixel of the tile) for tiles [t0, t1).  Uniform across the CTA.
template <class F>
__device__ __forceinline__ void for_each_tile(const Img* img, int n, long long t0, long long t1, F&& f) {
  int lo = 0, hi = n - 1;                              // the last image with tile0 <= t0
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (img[mid].tile0 <= t0) lo = mid; else hi = mid - 1;
  }
  for (long long t = t0; t < t1; ++t) {
    while (lo + 1 < n && img[lo + 1].tile0 <= t) ++lo;
    f(img[lo], (int)((t - img[lo].tile0) * kTile));
  }
}

__device__ __forceinline__ void flush(const unsigned* hist, int nb, unsigned long long* counts) {
  __syncthreads();
  for (int i = threadIdx.x; i < nb; i += kThreads) {
    const unsigned v = hist[i];
    if (v) atomicAdd(counts + i, (unsigned long long)v);
  }
}

// Histogram layout (shared memory and the caller's counters), Tp = T + 1, K = num_cls:
//   [(K-1) x Tp] pixels with best class c (row c-1) and j thresholds below its value
//   [(K-1) x Tp] the same, restricted to gt == c
//   [Tp]         pixels with gt == 0, by j
//   [K + 1]      pixels with gt == g for g < K; the last bin counts valid gt >= K
__global__ void __launch_bounds__(kThreads) cam_label_counts_kernel(const __grid_constant__ CamParams p) {
  extern __shared__ unsigned hist[];
  const int K = p.K, T = p.T, Tp = T + 1;
  const int nb = (2 * K - 1) * Tp + K + 1;
  float* thr = reinterpret_cast<float*>(hist + nb);
  for (int i = threadIdx.x; i < nb; i += kThreads) hist[i] = 0u;
  for (int i = threadIdx.x; i < T; i += kThreads) thr[i] = p.thr[i];
  __syncthreads();
  unsigned* h_pred = hist;
  unsigned* h_tp = hist + (K - 1) * Tp;
  unsigned* h_bg = hist + 2 * (K - 1) * Tp;
  unsigned* h_gt = h_bg + Tp;
  int step = 1;
  while (2 * step <= T) step *= 2;
  const int lane = threadIdx.x & 31;
  const long long t0 = (long long)blockIdx.x * p.tiles_per_cta, t1 = min(t0 + p.tiles_per_cta, p.total_tiles);

  for_each_tile(p.img, p.num_images, t0, t1, [&](const Img& im, int base) {
    const int end = (int)min((long long)base + kTile, im.npix) - base - threadIdx.x;    // pixel k is in range when k*kThreads < end
    const unsigned char* gt = p.gt + im.off + base + threadIdx.x;
    const float* cams = p.cams + base + threadIdx.x;
    const Plane* pl = p.planes + im.plane0;
    const int np = (int)im.nplanes;
    // first maximum over classes 1..K-1 in class order, absent classes reading 0; a NaN wins and stops the search
    // (np.argmax).  best = -inf with bc = the first candidate: a plane of -inf everywhere keeps the first class.
    // Every load of a plane (and of the ground truth) is issued for all kPer pixels of the thread before they are used.
    float best[kPer];
    int bc[kPer], g[kPer];
#pragma unroll
    for (int k = 0; k < kPer; ++k) {
      best[k] = -INFINITY;
      bc[k] = (int)im.first_label;
      g[k] = k * kThreads < end ? __ldg(gt + k * kThreads) : 255;
    }
    auto consider = [&](int k, float v, int lab) {
      if (best[k] == best[k] && (v != v || v > best[k])) {
        best[k] = v;
        bc[k] = lab;
      }
    };
    int z = (int)im.zero_label;
    for (int q = 0; q < np; ++q) {
      const int lab = (int)__ldg(&pl[q].label);
      const float* src = cams + __ldg(&pl[q].off);
      if (z < lab) {
#pragma unroll
        for (int k = 0; k < kPer; ++k) consider(k, 0.f, z);
        z = K;
      }
      float v[kPer];
#pragma unroll
      for (int k = 0; k < kPer; ++k) v[k] = k * kThreads < end ? __ldg(src + k * kThreads) : 0.f;
#pragma unroll
      for (int k = 0; k < kPer; ++k) consider(k, v[k], lab);
    }
    if (z < K) {
#pragma unroll
      for (int k = 0; k < kPer; ++k) consider(k, 0.f, z);
    }
#pragma unroll
    for (int k = 0; k < kPer; ++k) {                   // whole warps reach __match_any_sync
      unsigned key = 0xffffffffu;                      // no bin (bit 31 is never set in a real key)
      if (g[k] != 255) {                               // out-of-range pixels read 255 too
        int j = 0;                                     // thresholds strictly below best (a NaN is above all of them)
        if (best[k] != best[k]) {
          j = T;
        } else {
          for (int s = step; s > 0; s >>= 1)
            if (j + s <= T && thr[j + s - 1] < best[k]) j += s;
        }
        key = (unsigned)bc[k] << 21 | (unsigned)j << 8 | (unsigned)g[k];
      }
      const unsigned peers = __match_any_sync(0xffffffffu, key);
      if (key != 0xffffffffu && lane == __ffs(peers) - 1) {
        const unsigned n = __popc(peers);
        const int c = (int)(key >> 21), j = (int)((key >> 8) & 0x1fffu), gk = (int)(key & 0xffu);
        if (c > 0) {                                   // K = 1: no class, every pixel is background
          atomicAdd(h_pred + (c - 1) * Tp + j, n);
          if (gk == c) atomicAdd(h_tp + (c - 1) * Tp + j, n);
        }
        if (gk == 0) atomicAdd(h_bg + j, n);
        atomicAdd(h_gt + min(gk, K), n);
      }
    }
  });
  flush(hist, nb, p.counts);
}

// Label-map mode: counts [3][K] = P (pred == c), T (gt == c), TP (both) over pixels with gt != 255, labels < K.
__global__ void __launch_bounds__(kThreads) label_map_counts_kernel(const __grid_constant__ MapParams p) {
  __shared__ unsigned hist[3 * 255];
  const int K = p.K;
  for (int i = threadIdx.x; i < 3 * K; i += kThreads) hist[i] = 0u;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const long long t0 = (long long)blockIdx.x * p.tiles_per_cta, t1 = min(t0 + p.tiles_per_cta, p.total_tiles);
  for_each_tile(p.img, p.num_images, t0, t1, [&](const Img& im, int base) {
    const int end = (int)min((long long)base + kTile, im.npix) - base - threadIdx.x;
    const unsigned char* gt = p.gt + im.off + base + threadIdx.x;
    const unsigned char* pred = p.pred + im.off + base + threadIdx.x;
    int g[kPer], pr[kPer];
#pragma unroll
    for (int k = 0; k < kPer; ++k) {
      const bool in = k * kThreads < end;
      g[k] = in ? __ldg(gt + k * kThreads) : 255;
      pr[k] = in ? __ldg(pred + k * kThreads) : 0;
    }
#pragma unroll
    for (int k = 0; k < kPer; ++k) {
      const unsigned key = g[k] != 255 ? (unsigned)pr[k] << 8 | (unsigned)g[k] : 0xffffffffu;
      const unsigned peers = __match_any_sync(0xffffffffu, key);
      if (key != 0xffffffffu && lane == __ffs(peers) - 1) {
        const unsigned n = __popc(peers);
        if (pr[k] < K) atomicAdd(hist + pr[k], n);
        if (g[k] < K) {
          atomicAdd(hist + K + g[k], n);
          if (pr[k] == g[k]) atomicAdd(hist + 2 * K + g[k], n);
        }
      }
    }
  });
  flush(hist, 3 * K, p.counts);
}

size_t workspace_bytes_for(long long num_images, long long num_planes, long long T) {
  return (size_t)num_images * sizeof(Img) + (size_t)num_planes * sizeof(Plane) + (size_t)T * sizeof(float);
}

// Validates the image table {off, rows, cols} against a buffer of `elems` bytes and fills rows' off / npix / tile0.
int image_rows(const char* fn, const long long* images_host, int num_images, long long elems, std::vector<Img>& img,
               long long& tiles) {
  img.assign(num_images, Img{});
  tiles = 0;
  for (int i = 0; i < num_images; ++i) {
    const long long off = images_host[3 * i], rows = images_host[3 * i + 1], cols = images_host[3 * i + 2];
    ACR_REQUIRE(rows >= 1 && cols >= 1 && rows < (1LL << 31) && cols < (1LL << 31) && rows * cols < (1LL << 31), ACR_E_INVAL,
                "%s: image %d: bad size %lld x %lld (1 <= rows*cols < 2^31)", fn, i, rows, cols);
    ACR_REQUIRE(off >= 0 && off <= elems && rows * cols <= elems - off, ACR_E_INVAL,
                "%s: image %d overflows the %lld-element label buffer", fn, i, elems);
    img[i].off = off;
    img[i].npix = rows * cols;
    img[i].tile0 = tiles;
    tiles += (rows * cols + kTile - 1) / kTile;
  }
  return 0;
}

template <class Kernel>
int grid_for(Kernel kernel, size_t smem, long long tiles, long long& tiles_per_cta, long long& grid) {
  int dev = 0, sms = 0, per_sm = 0;
  ACR_CUDA(cudaGetDevice(&dev));
  ACR_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  ACR_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kThreads, smem));
  const long long ctas = (long long)std::max(1, sms) * std::max(1, per_sm);
  tiles_per_cta = std::min(kMaxTilesPerCta, (tiles + ctas - 1) / ctas);
  grid = (tiles + tiles_per_cta - 1) / tiles_per_cta;
  ACR_REQUIRE(grid <= INT32_MAX, ACR_E_INVAL, "label counts: %lld tiles are too many for one launch", tiles);
  return 0;
}

}  // namespace

extern "C" size_t acr_label_counts_workspace(int num_images, int num_planes, int num_thresholds) {
  if (num_images < 0 || num_planes < 0 || num_thresholds < 0) return 0;
  return workspace_bytes_for(num_images, num_planes, num_thresholds);
}

extern "C" int acr_cam_label_counts(const float* cams, long long cam_elems, const long long* planes_host, int num_planes,
                                    const unsigned char* gt, long long gt_elems, const long long* images_host, int num_images,
                                    const double* thresholds_host, int num_thresholds, int num_cls, long long* counts,
                                    void* workspace, size_t workspace_bytes, void* stream) {
  const char* fn = "acr_cam_label_counts";
  ACR_REQUIRE(gt && images_host && thresholds_host && counts && workspace, ACR_E_INVAL, "%s: null pointer", fn);
  ACR_REQUIRE(num_planes == 0 || (cams && planes_host), ACR_E_INVAL, "%s: null pointer", fn);
  ACR_REQUIRE(num_cls >= 1 && num_cls <= 255, ACR_E_INVAL, "%s: num_cls %d (1..255)", fn, num_cls);
  ACR_REQUIRE(num_images >= 0 && num_planes >= 0 && cam_elems >= 0 && gt_elems >= 0, ACR_E_INVAL, "%s: negative count", fn);
  ACR_REQUIRE(num_thresholds >= 1 && num_thresholds <= kMaxThresholds, ACR_E_INVAL, "%s: %d thresholds (1..%d)", fn,
              num_thresholds, kMaxThresholds);
  const int K = num_cls, T = num_thresholds;
  const size_t hist = (size_t)(2 * K - 1) * (T + 1) * 4 + 4 * (size_t)K;
  ACR_REQUIRE(hist <= kMaxHist, ACR_E_INVAL, "%s: histograms of %zu bytes for %d classes and %d thresholds exceed %zu bytes of "
              "shared memory", fn, hist, K, T, kMaxHist);
  std::vector<float> thr(T);
  for (int t = 0; t < T; ++t) {
    thr[t] = (float)thresholds_host[t];
    ACR_REQUIRE(std::isfinite(thresholds_host[t]) && std::isfinite(thr[t]), ACR_E_INVAL,
                "%s: threshold %d is not finite in float32", fn, t);
    ACR_REQUIRE(t == 0 || thr[t] >= thr[t - 1], ACR_E_INVAL, "%s: thresholds descend at %d (after float32 rounding)", fn, t);
  }
  std::vector<Img> img;
  long long tiles = 0;
  if (int e = image_rows(fn, images_host, num_images, gt_elems, img, tiles)) return e;

  // planes sorted by (image, class); a repeated class, a class >= K-1 or a plane outside the buffer is rejected
  std::vector<int> order(num_planes);
  for (int i = 0; i < num_planes; ++i) {
    const long long off = planes_host[3 * i], image = planes_host[3 * i + 1], cls = planes_host[3 * i + 2];
    ACR_REQUIRE(image >= 0 && image < num_images, ACR_E_INVAL, "%s: plane %d: image %lld out of range", fn, i, image);
    ACR_REQUIRE(cls >= 0 && cls < K - 1, ACR_E_INVAL, "%s: plane %d: class %lld out of range (0..%d)", fn, i, cls, K - 2);
    ACR_REQUIRE(off >= 0 && off <= cam_elems && img[image].npix <= cam_elems - off, ACR_E_INVAL,
                "%s: plane %d overflows the %lld-element CAM buffer", fn, i, cam_elems);
    order[i] = i;
  }
  std::sort(order.begin(), order.end(), [&](int a, int b) {
    const long long ia = planes_host[3 * a + 1], ib = planes_host[3 * b + 1];
    return ia != ib ? ia < ib : planes_host[3 * a + 2] < planes_host[3 * b + 2];
  });
  std::vector<Plane> planes(num_planes);
  for (int r = 0; r < num_planes; ++r) {
    const long long* d = planes_host + 3 * (long long)order[r];
    planes[r] = {d[0], d[2] + 1};
    if (r > 0) {
      const long long* q = planes_host + 3 * (long long)order[r - 1];
      ACR_REQUIRE(q[1] != d[1] || q[2] != d[2], ACR_E_INVAL, "%s: image %lld has two planes of class %lld", fn, d[1], d[2]);
    }
  }
  for (int r = 0, i = 0; i < num_images; ++i) {
    img[i].plane0 = r;
    long long zero = 1;                                // first label without a plane (K: none)
    while (r < num_planes && planes_host[3 * (long long)order[r] + 1] == i) {
      if (planes[r].label == zero) ++zero;
      ++r;
    }
    img[i].nplanes = r - img[i].plane0;
    img[i].zero_label = std::min<long long>(zero, K);
    img[i].first_label = img[i].nplanes ? std::min(zero, planes[img[i].plane0].label) : zero;
    if (K == 1) img[i].first_label = 0;                // no class at all
  }

  const size_t need = workspace_bytes_for(num_images, num_planes, T);
  ACR_REQUIRE(workspace_bytes >= need, ACR_E_NOMEM, "%s: workspace of %zu bytes needed", fn, need);
  ACR_REQUIRE(((uintptr_t)workspace & 7) == 0 && ((uintptr_t)counts & 7) == 0, ACR_E_ALIGN,
              "%s: workspace and counts must be 8-byte aligned", fn);
  if (tiles == 0) return 0;
  ACR_REQUIRE(acr_device_is_sm100(), ACR_E_NOSM100, "%s: needs an sm_100 device", fn);

  std::vector<char> table(need);
  char* w = table.data();
  memcpy(w, img.data(), img.size() * sizeof(Img));
  memcpy(w + img.size() * sizeof(Img), planes.data(), planes.size() * sizeof(Plane));
  memcpy(w + img.size() * sizeof(Img) + planes.size() * sizeof(Plane), thr.data(), thr.size() * sizeof(float));
  const cudaStream_t st = (cudaStream_t)stream;
  ACR_CUDA(cudaMemcpyAsync(workspace, table.data(), need, cudaMemcpyHostToDevice, st));    // staged before it returns

  const size_t smem = hist + 4 + (size_t)T * sizeof(float);
  static bool attr_set[64] = {false};
  if (int e = acr_attn::set_max_smem(cam_label_counts_kernel, kMaxSmem, attr_set)) return e;
  CamParams p = {};
  p.cams = cams;
  p.gt = gt;
  p.counts = reinterpret_cast<unsigned long long*>(counts);
  p.img = reinterpret_cast<const Img*>(workspace);
  p.planes = reinterpret_cast<const Plane*>((char*)workspace + img.size() * sizeof(Img));
  p.thr = reinterpret_cast<const float*>((char*)workspace + img.size() * sizeof(Img) + planes.size() * sizeof(Plane));
  p.num_images = num_images;
  p.K = K;
  p.T = T;
  p.total_tiles = tiles;
  long long grid = 0;
  if (int e = grid_for(cam_label_counts_kernel, smem, tiles, p.tiles_per_cta, grid)) return e;
  acr::KernelTimer kt_("cam_label_counts_kernel", st);
  cam_label_counts_kernel<<<(unsigned)grid, kThreads, smem, st>>>(p);
  return acr::check_launch("cam_label_counts_kernel");
}

extern "C" int acr_label_map_counts(const unsigned char* pred, const unsigned char* gt, long long elems, const long long* images_host,
                                    int num_images, int num_cls, long long* counts, void* workspace, size_t workspace_bytes,
                                    void* stream) {
  const char* fn = "acr_label_map_counts";
  ACR_REQUIRE(pred && gt && images_host && counts && workspace, ACR_E_INVAL, "%s: null pointer", fn);
  ACR_REQUIRE(num_cls >= 1 && num_cls <= 255, ACR_E_INVAL, "%s: num_cls %d (1..255)", fn, num_cls);
  ACR_REQUIRE(num_images >= 0 && elems >= 0, ACR_E_INVAL, "%s: negative count", fn);
  std::vector<Img> img;
  long long tiles = 0;
  if (int e = image_rows(fn, images_host, num_images, elems, img, tiles)) return e;
  const size_t need = workspace_bytes_for(num_images, 0, 0);
  ACR_REQUIRE(workspace_bytes >= need, ACR_E_NOMEM, "%s: workspace of %zu bytes needed", fn, need);
  ACR_REQUIRE(((uintptr_t)workspace & 7) == 0 && ((uintptr_t)counts & 7) == 0, ACR_E_ALIGN,
              "%s: workspace and counts must be 8-byte aligned", fn);
  if (tiles == 0) return 0;
  ACR_REQUIRE(acr_device_is_sm100(), ACR_E_NOSM100, "%s: needs an sm_100 device", fn);
  const cudaStream_t st = (cudaStream_t)stream;
  ACR_CUDA(cudaMemcpyAsync(workspace, img.data(), need, cudaMemcpyHostToDevice, st));
  MapParams p = {};
  p.pred = pred;
  p.gt = gt;
  p.counts = reinterpret_cast<unsigned long long*>(counts);
  p.img = reinterpret_cast<const Img*>(workspace);
  p.num_images = num_images;
  p.K = num_cls;
  p.total_tiles = tiles;
  long long grid = 0;
  if (int e = grid_for(label_map_counts_kernel, 0, tiles, p.tiles_per_cta, grid)) return e;
  acr::KernelTimer kt_("label_map_counts_kernel", st);
  label_map_counts_kernel<<<(unsigned)grid, kThreads, 0, st>>>(p);
  return acr::check_launch("label_map_counts_kernel");
}
