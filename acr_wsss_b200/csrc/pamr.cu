// (a10) PAMR -- pixel-adaptive mask refinement.  Reference: pamr.py:10-144.
//
// The reference builds [B,K,9D,H,W] / [B,K,8D,H,W] / [B,C,8D,H,W] intermediates with one-hot dilated
// conv2d calls (pamr.py:51-52) -- 810 MB per iteration at C=21, D=6, 448x448.  Here:
//   1. pamr_upsample_kernel     : bilinear, align_corners=True (pamr.py:126), into the ping buffer;
//   2. pamr_affinity_reg_kernel : per pixel, the 8D softmax weights w[b,n,y,x] (std over the 9D samples,
//                                 -|xc-xn|/(1e-8+0.1 std), mean over the K image channels, softmax over n), in registers;
//   3. num_iter iterations of mask[b,c,y,x] <- sum_n w[b,n,y,x] * mask[b,c,clamp(y+dy),clamp(x+dx)], by
//        pamr_iter_tma2_kernel (D <= 6 and every dilation <= kPamrHalo): TMA-fed shared-memory tiles, then
//                              pamr_pad_kernel refills the replicated ring of the result;
//        pamr_iter_kernel      (any other list): one thread per pixel, clamped loads through L1 / L2.
// Neighbour order per dilation is row-major over the 3x3 window without its centre (pamr.py:24-33);
// dilations are concatenated in list order (pamr.py:55); borders replicate (pamr.py:51).  Both iteration
// kernels add the taps in this order, so they produce bit-identical sums.
//
// Layout.  The ping / pong masks are [B*C][H + 2R][P]: R = kPamrHalo cells on every side of the image repeat its
// edge pixels, and the row pitch P is W + 2R rounded up to 4 floats, as TMA strides must be multiples of 16 bytes (the
// cells past W + 2R are never read).  The affinity weights are [B*8D][H][Wq] with Wq = W rounded up to 4.  The last
// iteration writes the caller's unpadded [B,C,H,W] output.
// Bandwidth-bound: algorithmic bytes = HW(4K + 32D) for step 2 and HW(32D + 8C) per iteration.
// The backward (acr_pamr_bwd, after acr_pamr_fwd_save kept the weights and every iterate) is at the end of the file.
#include "attn_tc.cuh"      // tc:: mbarrier / TMA helpers, acr_attn::get_encode_fn

namespace {

constexpr int kMaxDil = 8;
struct Dil { int d[kMaxDil]; int n; };

constexpr int kPamrHalo = 24;      // compile-time halo (largest dilation of the tiled path): keeps every LDS address an immediate
                                   // offset from one per-tap register (runtime strides cost 4 integer ops per tap)

int pad_pitch(int W) { return (W + 2 * kPamrHalo + 3) / 4 * 4; }
int wgt_pitch(int W) { return (W + 3) / 4 * 4; }
size_t wgt_bytes(int B, int nd, int H, int W) { return acr::align_up((size_t)B * 8 * nd * H * wgt_pitch(W) * sizeof(float), 256); }
size_t mask_bytes(int B, int C, int H, int W) {
  return acr::align_up((size_t)B * C * (H + 2 * kPamrHalo) * pad_pitch(W) * sizeof(float), 256);
}

// A mask in memory: pixel (0, 0) of plane 0, and the distances of rows and of planes, in floats.
struct MaskBuf { float* p; int pitch; long long plane; };

MaskBuf padded_mask(float* buf, int H, int W) {
  const int P = pad_pitch(W);
  return {buf + (long long)kPamrHalo * P + kPamrHalo, P, (long long)(H + 2 * kPamrHalo) * P};
}

__device__ __forceinline__ int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

__global__ void __launch_bounds__(256)
pamr_upsample_kernel(const float* __restrict__ src, int planes, int h, int w, int H, int W, int pad, int pitch, float* __restrict__ dst) {
  // dst: [planes, H + 2 pad, pitch]; the pad ring repeats the edge pixels
  const int Wp = W + 2 * pad, Hp = H + 2 * pad;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long total = (long long)planes * Hp * Wp;
  if (idx >= total) return;
  const long long row = idx / Wp;                                  // plane * Hp + padded row
  const int x = clampi((int)(idx % Wp) - pad, 0, W - 1);
  const int y = clampi((int)(row % Hp) - pad, 0, H - 1);
  const long long pl = row / Hp;
  const float sy = (H > 1) ? (float)(h - 1) / (float)(H - 1) : 0.f;
  const float sx = (W > 1) ? (float)(w - 1) / (float)(W - 1) : 0.f;
  const float fy = sy * (float)y, fx = sx * (float)x;
  const int y0 = min((int)fy, h - 1), x0 = min((int)fx, w - 1);
  const int y1 = min(y0 + 1, h - 1), x1 = min(x0 + 1, w - 1);
  const float ly = fy - (float)y0, lx = fx - (float)x0;
  const float hy = 1.f - ly, hx = 1.f - lx;
  const float* p = src + pl * h * w;
  const float v = hy * (hx * __ldg(p + y0 * w + x0) + lx * __ldg(p + y0 * w + x1)) +
                  ly * (hx * __ldg(p + y1 * w + x0) + lx * __ldg(p + y1 * w + x1));
  dst[row * pitch + idx % Wp] = v;
}

// One thread per pixel: the 9*ND samples of a channel and the 8*ND logits live in registers, and each weight plane is
// written exactly once.  wgt layout [B, 8*ND, H, wpitch].
// (Round-1 experiments with 4-pixel "quad" threads and with channel-outer / register-resident weights were 1.1-5x SLOWER
// than a scalar tap-outer kernel -- low occupancy and L1 thrashing across channel planes; see DESIGN.md.)
template <int ND>
__global__ void __launch_bounds__(128)
pamr_affinity_reg_kernel(const float* __restrict__ x, int K, int H, int W, Dil dil, int wpitch, float* __restrict__ wgt) {
  const int px = blockIdx.x * blockDim.x + threadIdx.x;
  const int py = blockIdx.y;
  const int b = blockIdx.z;
  if (px >= W) return;
  const long long HW = (long long)H * W;
  constexpr int NN = 8 * ND;
  float aff[NN];
#pragma unroll
  for (int n = 0; n < NN; ++n) aff[n] = 0.f;
  for (int k = 0; k < K; ++k) {
    const float* img = x + ((long long)b * K + k) * HW;
    float v[9 * ND];
    float sum = 0.f;
#pragma unroll
    for (int di = 0; di < ND; ++di) {
      const int d = dil.d[di];
#pragma unroll
      for (int t = 0; t < 9; ++t) {
        const int yy = clampi(py + (t / 3 - 1) * d, 0, H - 1), xx = clampi(px + (t % 3 - 1) * d, 0, W - 1);
        v[di * 9 + t] = __ldg(img + (long long)yy * W + xx);
        sum += v[di * 9 + t];
      }
    }
    const float mean = sum / (float)(9 * ND);
    float ss = 0.f;
#pragma unroll
    for (int i = 0; i < 9 * ND; ++i) { const float dv = v[i] - mean; ss += dv * dv; }
    const float sd = sqrtf(ss / (float)(9 * ND - 1));
    const float inv = 1.f / (1e-8f + 0.1f * sd);
    const float xc = v[4];
#pragma unroll
    for (int di = 0; di < ND; ++di)
#pragma unroll
      for (int t = 0; t < 9; ++t) {
        if (t == 4) continue;
        const int n = di * 8 + (t < 4 ? t : t - 1);
        aff[n] += -fabsf(xc - v[di * 9 + t]) * inv;
      }
  }
  const float invK = 1.f / (float)K;
  float m = -INFINITY;
#pragma unroll
  for (int n = 0; n < NN; ++n) { aff[n] *= invK; m = fmaxf(m, aff[n]); }
  float ssum = 0.f;
#pragma unroll
  for (int n = 0; n < NN; ++n) { aff[n] = expf(aff[n] - m); ssum += aff[n]; }
  const float invs = 1.f / ssum;
  const long long plane = (long long)H * wpitch;
  float* wp = wgt + (long long)b * NN * plane + (long long)py * wpitch + px;
#pragma unroll
  for (int n = 0; n < NN; ++n) wp[n * plane] = aff[n] * invs;
}

// Iteration for the dilation lists the tiled kernel below cannot serve (more than 6, or one beyond its halo): one thread per
// pixel and group of kIterCG channels, clamped taps through L1 / L2.  It reads the interior of the padded source only.
constexpr int kIterCG = 3, kIterTW = 32;                           // block = 32 x 8 pixels
__global__ void __launch_bounds__(256)
pamr_iter_kernel(const float* __restrict__ wgt, int wpitch, MaskBuf src, MaskBuf dst, int C, int H, int W, Dil dil, int groups) {
  const int px = blockIdx.x * kIterTW + (threadIdx.x % kIterTW);
  const int py = blockIdx.y * (256 / kIterTW) + (threadIdx.x / kIterTW);
  const int b = blockIdx.z / groups, g = blockIdx.z % groups;
  if (px >= W || py >= H) return;
  const long long wplane = (long long)H * wpitch;
  const int nn = 8 * dil.n;
  const float* wp = wgt + (long long)b * nn * wplane + (long long)py * wpitch + px;
  const int c0 = g * kIterCG;
  float acc[kIterCG];
#pragma unroll
  for (int c = 0; c < kIterCG; ++c) acc[c] = 0.f;
  const float* mb = src.p + ((long long)b * C + c0) * src.plane;
  int n = 0;
  for (int di = 0; di < dil.n; ++di) {
    const int d = dil.d[di];
#pragma unroll
    for (int t = 0; t < 9; ++t) {
      if (t == 4) continue;
      const int yy = clampi(py + (t / 3 - 1) * d, 0, H - 1), xx = clampi(px + (t % 3 - 1) * d, 0, W - 1);
      const float wv = __ldg(wp + n * wplane);
      const float* mp = mb + (long long)yy * src.pitch + xx;
#pragma unroll
      for (int c = 0; c < kIterCG; ++c)
        if (c0 + c < C) acc[c] = fmaf(wv, __ldg(mp + c * src.plane), acc[c]);
      ++n;
    }
  }
  float* op = dst.p + ((long long)b * C + c0) * dst.plane + (long long)py * dst.pitch + px;
#pragma unroll
  for (int c = 0; c < kIterCG; ++c)
    if (c0 + c < C) op[c * dst.plane] = acc[c];
}

// TMA-fed shared-memory tiles.  48 taps per output make the iteration a gather problem (808 MB of tap reads per iteration at
// cfg3, against 46 MB of compulsory HBM traffic).  A CTA owns a 32 x 16 output tile: the 8*ND weights of a thread's two pixels
// live in registers, the mask tile of kPamrCh channels with a halo of kPamrHalo arrives by cp.async.bulk.tensor from the
// replicate-padded source (so the tap loop has no clamps and no thread patches halos), and every tap is one conflict-free LDS +
// one FMA.  256 threads and a single 61 KB stage let TWO CTAs share an SM, so one CTA's prologue and TMA round trip run under
// the other's tap loop (ncu on a 32 x 32-tile, one-CTA-per-SM version: profiles/r02_ncu_refine_kernels.txt).
// Bound: one warp-wide LDS per clock per SM.
// (A persistent variant -- one CTA per SM walking over the work items with the TMA ring running across items -- was 40 %
// SLOWER: the per-item state pushed the 96 weight registers into local memory, profiles/r02_ncu_pamr_persistent.txt.  A
// one-pixel-per-thread variant -- 512 threads, 48 weights, two CTAs per SM at 64 registers -- spilt 56 of its 48+ live
// values and was 10 % slower than the two-pixel version.)
constexpr int kPamrTile = 32, kPamrTileH = 16;                     // output tile: 32 columns x 16 rows
constexpr int kPamrTS = kPamrTile + 2 * kPamrHalo;                 // 80 columns of a stage
constexpr int kPamrTSY = kPamrTileH + 2 * kPamrHalo;               // 64 rows of a stage
constexpr int kPamrCh = 3;                                         // channels per stage
constexpr int kPamrStage = kPamrCh * kPamrTSY * kPamrTS;           // floats per stage (61,440 B)
// The dilation list every caller of the reference uses (pamr.py default of the upstream PAMR, BASELINE configs[2]) as
// compile-time constants: every tap address becomes an immediate offset from ONE register.  With run-time dilations the tap
// loop carried ~8 integer instructions per tap next to its 6 LDS + 6 FFMA and the kernel was issue bound (ncu r02a: 61 % of
// the issue slots, ALU pipe 39 %, shared-memory pipe 45 %).
__host__ __device__ constexpr int std_dil(int i) { return i == 0 ? 1 : i == 1 ? 2 : i == 2 ? 4 : i == 3 ? 8 : i == 4 ? 12 : 24; }

// taps of NCH channels of the stage for this thread's two pixels (stage rows r and r + 8)
template <int ND, int NCH, bool STD>
__device__ __forceinline__ void pamr_taps(const float* __restrict__ t, int base, const Dil& dil, const float (&w0)[8 * ND], const float (&w1)[8 * ND],
                                          float (&a0)[kPamrCh], float (&a1)[kPamrCh]) {
  constexpr int TS = kPamrTS, per = kPamrTSY * kPamrTS;
#pragma unroll
  for (int c = 0; c < NCH; ++c) { a0[c] = 0.f; a1[c] = 0.f; }
#pragma unroll
  for (int di = 0; di < ND; ++di) {
    const int d = STD ? std_dil(di) : dil.d[di];
#pragma unroll
    for (int tp = 0; tp < 9; ++tp) {
      if (tp == 4) continue;
      const int n = di * 8 + (tp < 4 ? tp : tp - 1);
      const int off = base + (tp / 3 - 1) * d * TS + (tp % 3 - 1) * d;
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        a0[c] = fmaf(w0[n], t[c * per + off], a0[c]);
        a1[c] = fmaf(w1[n], t[c * per + off + 8 * TS], a1[c]);
      }
    }
  }
}

// One CTA per (tile, channel group of CG).  tmap_mask: the padded source; tmap_wgt: the weight planes.
template <int ND, int CG, bool STD>
__global__ void __launch_bounds__(256, 2)
pamr_iter_tma2_kernel(const __grid_constant__ CUtensorMap tmap_mask, const __grid_constant__ CUtensorMap tmap_wgt,
                      MaskBuf dst, int C, int H, int W, Dil dil, int groups) {
  // shared: first the 8*ND weight planes of this tile ([8*ND][16][32] floats, one TMA box: 96 loads per thread through the LSU queue
  // were the slowest part of the CTA), then -- once they sit in registers -- the mask stage [kPamrCh][TSY][TS]; then two mbarriers
  extern __shared__ __align__(128) float tile[];
  constexpr int TS = kPamrTS, R = kPamrHalo;
  constexpr int kWgtFloats = 8 * ND * kPamrTileH * kPamrTile;
  constexpr int kBufFloats = kWgtFloats > kPamrStage ? kWgtFloats : kPamrStage;
  uint64_t* full = reinterpret_cast<uint64_t*>(tile + kBufFloats);
  uint64_t* wfull = full + 1;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;         // 32 x 8 threads, two rows per thread (ty, ty + 8)
  const int x0 = blockIdx.x * kPamrTile, y0 = blockIdx.y * kPamrTileH;
  const int b = blockIdx.z / groups, g = blockIdx.z % groups;
  const int c0 = g * CG, cend = min(C, c0 + CG);
  const int nchunks = (cend - c0 + kPamrCh - 1) / kPamrCh;
  auto issue = [&](int k) {
    // padded coordinates: image pixel (x, y) sits at (x + R, y + R), so the box of tile (x0, y0) starts at (x0, y0)
    tc::mbar_arrive_expect_tx(full, kPamrStage * sizeof(float));
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
                     tc::smem_u32(tile)),
                 "l"(reinterpret_cast<uint64_t>(&tmap_mask)), "r"(tc::smem_u32(full)), "r"(x0), "r"(y0), "r"(b * C + c0 + k * kPamrCh)
                 : "memory");
  };
  if (threadIdx.x == 0) {
    tc::prefetch_tmap(&tmap_mask);
    tc::prefetch_tmap(&tmap_wgt);
    tc::mbar_init(full, 1);
    tc::mbar_init(wfull, 1);
    tc::fence_barrier_init();
    tc::mbar_arrive_expect_tx(wfull, kWgtFloats * sizeof(float));
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
                     tc::smem_u32(tile)),
                 "l"(reinterpret_cast<uint64_t>(&tmap_wgt)), "r"(tc::smem_u32(wfull)), "r"(x0), "r"(y0), "r"(b * 8 * ND)
                 : "memory");
  }
  const int px = x0 + tx, py0 = y0 + ty, py1 = y0 + ty + 8;
  const bool ok0 = px < W && py0 < H, ok1 = px < W && py1 < H;
  float w0[8 * ND], w1[8 * ND];
  __syncthreads();                                                 // barrier initialisation visible to every waiter
  tc::mbar_wait(wfull, 0);
#pragma unroll
  for (int n = 0; n < 8 * ND; ++n) {
    w0[n] = tile[(n * kPamrTileH + ty) * kPamrTile + tx];
    w1[n] = tile[(n * kPamrTileH + ty + 8) * kPamrTile + tx];
  }
  __syncthreads();                                                 // everyone holds its weights: the buffer becomes the mask stage
  if (threadIdx.x == 0) {
    tc::fence_proxy_async_smem();
    issue(0);
  }
  const int base = (ty + R) * TS + tx + R;
  for (int k = 0; k < nchunks; ++k) {
    tc::mbar_wait(full, k & 1);
    float a0[kPamrCh], a1[kPamrCh];
    const int nch = min(kPamrCh, cend - (c0 + k * kPamrCh));       // the last chunk of a group may hold fewer channels
    if (nch == kPamrCh) pamr_taps<ND, kPamrCh, STD>(tile, base, dil, w0, w1, a0, a1);
    else if (nch == 2) pamr_taps<ND, 2, STD>(tile, base, dil, w0, w1, a0, a1);
    else pamr_taps<ND, 1, STD>(tile, base, dil, w0, w1, a0, a1);
    __syncthreads();                                               // every thread is done with the stage
    if (threadIdx.x == 0 && k + 1 < nchunks) {
      tc::fence_proxy_async_smem();                                // generic-proxy reads of the stage before the async-proxy refill
      issue(k + 1);
    }
    float* op = dst.p + ((long long)b * C + c0 + k * kPamrCh) * dst.plane + px;
#pragma unroll
    for (int c = 0; c < kPamrCh; ++c) {
      if (c < nch) {
        if (ok0) op[c * dst.plane + (long long)py0 * dst.pitch] = a0[c];
        if (ok1) op[c * dst.plane + (long long)py1 * dst.pitch] = a1[c];
      }
    }
  }
}

// Ring of a padded mask buffer [planes, H + 2R, pitch]: every cell outside the image repeats the nearest image pixel
// (pamr.py:51 pads with 'replicate').  One thread per ring cell: 4 (H + W + 2R) R cells per plane.
__global__ void __launch_bounds__(256)
pamr_pad_kernel(float* __restrict__ buf, int planes, int H, int W, int pitch) {
  constexpr int R = kPamrHalo;
  const int Wp = W + 2 * R, Hp = H + 2 * R;
  const int top = R * Wp;                                          // cells of the R rows above (and below) the image
  const int ring = 2 * top + 2 * R * H;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)planes * ring) return;
  const int e = (int)(idx % ring);
  float* plane = buf + (idx / ring) * (long long)Hp * pitch;
  int yp, xp;
  if (e < top) { yp = e / Wp; xp = e - yp * Wp; }
  else if (e < 2 * top) { const int q = e - top; yp = R + H + q / Wp; xp = q % Wp; }
  else { const int q = e - 2 * top; yp = R + q / (2 * R); const int c = q % (2 * R); xp = c < R ? c : W + c; }
  const int ys = clampi(yp, R, R + H - 1), xs = clampi(xp, R, R + W - 1);
  plane[(long long)yp * pitch + xp] = plane[(long long)ys * pitch + xs];
}

// fp32 tensor map over `planes` planes of h rows of w floats, rows `pitch` floats apart (pitch % 4 == 0); cells beyond the
// logical extents read as zero.
int make_plane_tmap(CUtensorMap* m, const float* base, int w, int h, int planes, int pitch, int box_w, int box_h, int box_planes) {
  acr_attn::EncodeTiledFn fn = acr_attn::get_encode_fn();
  ACR_REQUIRE(fn != nullptr, ACR_E_NOSM100, "cuTensorMapEncodeTiled unavailable");
  cuuint64_t dims[3] = {(cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)planes};
  cuuint64_t strides[2] = {(cuuint64_t)pitch * 4, (cuuint64_t)h * pitch * 4};
  cuuint32_t box[3] = {(cuuint32_t)box_w, (cuuint32_t)box_h, (cuuint32_t)box_planes};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  ACR_REQUIRE(r == CUDA_SUCCESS, ACR_E_INVAL, "cuTensorMapEncodeTiled failed (%d)", (int)r);
  return 0;
}

template <int ND, int CG, bool STD>
int launch_iter_tma2(const CUtensorMap& tmap, const CUtensorMap& tmap_wgt, const MaskBuf& dst, int B, int C, int H, int W, const Dil& dil,
                     cudaStream_t st) {
  const int groups = (C + CG - 1) / CG;
  constexpr size_t wfl = (size_t)8 * ND * kPamrTileH * kPamrTile;
  const size_t smem = (wfl > (size_t)kPamrStage ? wfl : (size_t)kPamrStage) * sizeof(float) + 64;
  static bool attr_set[64] = {false};
  if (int e = acr_attn::set_max_smem(pamr_iter_tma2_kernel<ND, CG, STD>, smem, attr_set)) return e;
  dim3 grid((W + kPamrTile - 1) / kPamrTile, (H + kPamrTileH - 1) / kPamrTileH, B * groups);
  pamr_iter_tma2_kernel<ND, CG, STD><<<grid, 256, smem, st>>>(tmap, tmap_wgt, dst, C, H, W, dil, groups);
  return acr::check_launch("pamr_iter_tma2_kernel");
}

template <int ND>
int launch_affinity_reg(const float* x, int B, int K, int H, int W, const Dil& dil, float* wgt, cudaStream_t st) {
  dim3 grid((W + 127) / 128, H, B);
  pamr_affinity_reg_kernel<ND><<<grid, 128, 0, st>>>(x, K, H, W, dil, wgt_pitch(W), wgt);
  return acr::check_launch("pamr_affinity_reg_kernel");
}

// num_iter >= 1 iterations starting from the padded ping buffer; the last one goes to `out`.  With slot_stride == 0 the
// intermediate results alternate between pong and ping; otherwise iterate t (1 <= t < num_iter) keeps its own padded buffer at
// ping + t * slot_stride bytes, so that the backward finds M_0 .. M_{num_iter-1}.  Both modes launch the same kernels on the same
// values, so their outputs are bitwise equal.
int pamr_iterate(const float* wgt, float* ping, float* pong, size_t slot_stride, float* out, int B, int C, int H, int W, const Dil& dil,
                 int num_iter, cudaStream_t st) {
  int maxd = 0;
  for (int i = 0; i < dil.n; ++i) maxd = dil.d[i] > maxd ? dil.d[i] : maxd;
  const bool tiled = dil.n <= 6 && maxd <= kPamrHalo;
  bool std6 = dil.n == 6;
  for (int i = 0; i < 6 && std6; ++i) std6 = dil.d[i] == std_dil(i);
  const int R = kPamrHalo, P = pad_pitch(W);
  auto slot = [&](int i) { return slot_stride ? (float*)((char*)ping + i * slot_stride) : (i & 1 ? pong : ping); };
  CUtensorMap tm_ping, tm_pong, tm_wgt;
  if (tiled) {
    if (!slot_stride) {
      if (int e = make_plane_tmap(&tm_ping, ping, W + 2 * R, H + 2 * R, B * C, P, kPamrTS, kPamrTSY, kPamrCh)) return e;
      if (int e = make_plane_tmap(&tm_pong, pong, W + 2 * R, H + 2 * R, B * C, P, kPamrTS, kPamrTSY, kPamrCh)) return e;
    }
    // one box = the 8 * nd weight planes of a 32 x 16 tile
    if (int e = make_plane_tmap(&tm_wgt, wgt, W, H, B * 8 * dil.n, wgt_pitch(W), kPamrTile, kPamrTileH, 8 * dil.n)) return e;
  }
  const MaskBuf m_out = {out, W, (long long)H * W};
  for (int it = 0; it < num_iter; ++it) {
    const bool last = it == num_iter - 1;
    const bool from_ping = !(it & 1);
    const MaskBuf dst = last ? m_out : padded_mask(slot(it + 1), H, W);
    int e = 0;
    if (tiled) {
      CUtensorMap tm_slot;
      if (slot_stride)
        if (int e2 = make_plane_tmap(&tm_slot, slot(it), W + 2 * R, H + 2 * R, B * C, P, kPamrTS, kPamrTSY, kPamrCh)) return e2;
      const CUtensorMap& tm = slot_stride ? tm_slot : (from_ping ? tm_ping : tm_pong);
      // channel groups of 21: the 96 weight loads per thread at the head of a CTA cost about as much as the taps of 7 channels, so
      // they are amortised over three times as many (measured at 448 x 448, C = 21: 693 -> 642 us for one image, 4708 -> 3651 us
      // for eight; C = 81: 2237 -> 1737 us).
      if (std6) {
        e = launch_iter_tma2<6, 21, true>(tm, tm_wgt, dst, B, C, H, W, dil, st);
      } else {
        switch (dil.n) {
          case 1: e = launch_iter_tma2<1, 7, false>(tm, tm_wgt, dst, B, C, H, W, dil, st); break;
          case 2: e = launch_iter_tma2<2, 7, false>(tm, tm_wgt, dst, B, C, H, W, dil, st); break;
          case 3: e = launch_iter_tma2<3, 7, false>(tm, tm_wgt, dst, B, C, H, W, dil, st); break;
          case 4: e = launch_iter_tma2<4, 7, false>(tm, tm_wgt, dst, B, C, H, W, dil, st); break;
          case 5: e = launch_iter_tma2<5, 7, false>(tm, tm_wgt, dst, B, C, H, W, dil, st); break;
          default: e = launch_iter_tma2<6, 7, false>(tm, tm_wgt, dst, B, C, H, W, dil, st); break;
        }
      }
      if (e) return e;
      if (!last) {
        const long long cells = (long long)B * C * (2 * R * (W + 2 * R) + 2 * R * H);
        pamr_pad_kernel<<<(unsigned)((cells + 255) / 256), 256, 0, st>>>(slot(it + 1), B * C, H, W, P);
        if (int e2 = acr::check_launch("pamr_pad_kernel")) return e2;
      }
    } else {
      // clamped taps read only the interior of the source, so the ring of the destination is left unfilled
      const int groups = (C + kIterCG - 1) / kIterCG;
      dim3 grid((W + kIterTW - 1) / kIterTW, (H + 256 / kIterTW - 1) / (256 / kIterTW), B * groups);
      pamr_iter_kernel<<<grid, 256, 0, st>>>(wgt, wgt_pitch(W), padded_mask(slot(it), H, W), dst, C, H, W, dil, groups);
      if (int e2 = acr::check_launch("pamr_iter_kernel")) return e2;
    }
  }
  return 0;
}

// ------------------------------------------------------------------------------------------------------------------------------
// Backward.  Every kernel is a gather with a fixed summation order (no atomics), so results are bitwise reproducible and an
// image's gradients do not depend on the rest of its batch.  The forward's taps read clamp(p + o_n); their adjoints collect,
// at pixel q, every (p, n) with clamp(p + o_n) = q.  Along one axis those p form the interval below: the pixel q - o, and on the
// two edge rows / columns also every pixel whose tap the replicate padding folded onto them.

// [lo, hi] (empty when lo > hi) = the p in [0, n) with clamp(p + o, 0, n - 1) == q
__device__ __forceinline__ void tap_sources(int q, int o, int n, int& lo, int& hi) {
  lo = q == 0 ? 0 : max(q - o, 0);
  hi = q == n - 1 ? n - 1 : min(q - o, n - 1);
}

// Adjoint of one iteration: gout[q, c] = sum over (p, n) with clamp(p + o_n) = q of w[p, n] * g[p, c].  g / gout are unpadded
// [B*C][H][W]; one thread per pixel and group of kIterCG channels, taps in the forward's order.
__global__ void __launch_bounds__(256)
pamr_iter_bwd_kernel(const float* __restrict__ wgt, int wpitch, const float* __restrict__ g, float* __restrict__ gout, int C, int H, int W,
                     Dil dil, int groups) {
  const int px = blockIdx.x * kIterTW + (threadIdx.x % kIterTW);
  const int py = blockIdx.y * (256 / kIterTW) + (threadIdx.x / kIterTW);
  const int b = blockIdx.z / groups, gi = blockIdx.z % groups;
  if (px >= W || py >= H) return;
  const long long HW = (long long)H * W, wplane = (long long)H * wpitch;
  const int c0 = gi * kIterCG;
  const float* wb = wgt + (long long)b * 8 * dil.n * wplane;
  const float* gb = g + ((long long)b * C + c0) * HW;
  float acc[kIterCG];
#pragma unroll
  for (int c = 0; c < kIterCG; ++c) acc[c] = 0.f;
  int n = 0;
  for (int di = 0; di < dil.n; ++di) {
    const int d = dil.d[di];
#pragma unroll
    for (int t = 0; t < 9; ++t) {
      if (t == 4) continue;
      int ylo, yhi, xlo, xhi;
      tap_sources(py, (t / 3 - 1) * d, H, ylo, yhi);
      tap_sources(px, (t % 3 - 1) * d, W, xlo, xhi);
      const float* wp = wb + n * wplane;
      for (int yy = ylo; yy <= yhi; ++yy)
        for (int xx = xlo; xx <= xhi; ++xx) {
          const float wv = __ldg(wp + (long long)yy * wpitch + xx);
          const float* gp = gb + (long long)yy * W + xx;
#pragma unroll
          for (int c = 0; c < kIterCG; ++c)
            if (c0 + c < C) acc[c] = fmaf(wv, __ldg(gp + c * HW), acc[c]);
        }
      ++n;
    }
  }
  float* op = gout + ((long long)b * C + c0) * HW + (long long)py * W + px;
#pragma unroll
  for (int c = 0; c < kIterCG; ++c)
    if (c0 + c < C) op[c * HW] = acc[c];
}

// Gradient of the weights from one iteration: dw[p, n] (+)= sum_c g[p, c] * m[clamp(p + o_n), c], the forward's taps with the
// channel sum inside the thread.  m: the saved padded iterate M_{t-1} (interior read through clamps); dw: [B, 8*ND, H, wpitch].
template <int ND>
__global__ void __launch_bounds__(128)
pamr_wgrad_kernel(const float* __restrict__ g, MaskBuf m, int C, int H, int W, Dil dil, int wpitch, int first, float* __restrict__ dw) {
  const int px = blockIdx.x * blockDim.x + threadIdx.x;
  const int py = blockIdx.y;
  const int b = blockIdx.z;
  if (px >= W) return;
  constexpr int NN = 8 * ND;
  const long long HW = (long long)H * W;
  float acc[NN];
#pragma unroll
  for (int n = 0; n < NN; ++n) acc[n] = 0.f;
  for (int c = 0; c < C; ++c) {
    const float gv = __ldg(g + ((long long)b * C + c) * HW + (long long)py * W + px);
    const float* mp = m.p + ((long long)b * C + c) * m.plane;
#pragma unroll
    for (int di = 0; di < ND; ++di) {
      const int d = dil.d[di];
#pragma unroll
      for (int t = 0; t < 9; ++t) {
        if (t == 4) continue;
        const int n = di * 8 + (t < 4 ? t : t - 1);
        const int yy = clampi(py + (t / 3 - 1) * d, 0, H - 1), xx = clampi(px + (t % 3 - 1) * d, 0, W - 1);
        acc[n] = fmaf(gv, __ldg(mp + (long long)yy * m.pitch + xx), acc[n]);
      }
    }
  }
  const long long plane = (long long)H * wpitch;
  float* wp = dw + (long long)b * NN * plane + (long long)py * wpitch + px;
#pragma unroll
  for (int n = 0; n < NN; ++n) wp[n * plane] = first ? acc[n] : wp[n * plane] + acc[n];
}

// Softmax and affinity backward, one thread per pixel p.  In: dw = dL/dw.  Out: dw becomes da = w * (dw - sum_m w dw), and per
// image channel k, stats [B, 4K, H, W] receives the four per-pixel factors the image gradient gathers:
//   A = r / K, f = dsigma / ((9D - 1) sigma) (0 where sigma = 0, as torch's std backward), the sample mean, and cen = the
// gradient of x_k(p) through the pixel's own centre taps: sum_n -da_k r sign(x_c - x_n) + D f (x_c - mean).
// The samples, mean, std and r are recomputed exactly as pamr_affinity_reg_kernel computes them.
template <int ND>
__global__ void __launch_bounds__(128)
pamr_affinity_bwd_kernel(const float* __restrict__ x, const float* __restrict__ wgt, int K, int H, int W, Dil dil, int wpitch,
                         float* __restrict__ dw, float* __restrict__ stats) {
  const int px = blockIdx.x * blockDim.x + threadIdx.x;
  const int py = blockIdx.y;
  const int b = blockIdx.z;
  if (px >= W) return;
  constexpr int NN = 8 * ND;
  const long long HW = (long long)H * W, pix = (long long)py * W + px;
  const long long plane = (long long)H * wpitch;
  const float* wp = wgt + (long long)b * NN * plane + (long long)py * wpitch + px;
  float* dp = dw + (long long)b * NN * plane + (long long)py * wpitch + px;
  float s = 0.f;
#pragma unroll
  for (int n = 0; n < NN; ++n) s = fmaf(wp[n * plane], dp[n * plane], s);
  float da[NN];
#pragma unroll
  for (int n = 0; n < NN; ++n) {
    da[n] = wp[n * plane] * (dp[n * plane] - s);
    dp[n * plane] = da[n];
  }
  const float invK = 1.f / (float)K;
  for (int k = 0; k < K; ++k) {
    const float* img = x + ((long long)b * K + k) * HW;
    float v[9 * ND];
    float sum = 0.f;
#pragma unroll
    for (int di = 0; di < ND; ++di) {
      const int d = dil.d[di];
#pragma unroll
      for (int t = 0; t < 9; ++t) {
        const int yy = clampi(py + (t / 3 - 1) * d, 0, H - 1), xx = clampi(px + (t % 3 - 1) * d, 0, W - 1);
        v[di * 9 + t] = __ldg(img + (long long)yy * W + xx);
        sum += v[di * 9 + t];
      }
    }
    const float mean = sum / (float)(9 * ND);
    float ss = 0.f;
#pragma unroll
    for (int i = 0; i < 9 * ND; ++i) { const float dv = v[i] - mean; ss += dv * dv; }
    const float sd = sqrtf(ss / (float)(9 * ND - 1));
    const float inv = 1.f / (1e-8f + 0.1f * sd);
    const float xc = v[4];
    float dr = 0.f, sg = 0.f;                                      // dL/dr, and sum_n da_n sign(x_c - x_n)
#pragma unroll
    for (int di = 0; di < ND; ++di)
#pragma unroll
      for (int t = 0; t < 9; ++t) {
        if (t == 4) continue;
        const int n = di * 8 + (t < 4 ? t : t - 1);
        const float u = xc - v[di * 9 + t];
        dr -= da[n] * fabsf(u);
        sg += u > 0.f ? da[n] : (u < 0.f ? -da[n] : 0.f);
      }
    dr *= invK;
    const float dsd = -0.1f * inv * inv * dr;
    const float f = sd > 0.f ? dsd / ((float)(9 * ND - 1) * sd) : 0.f;
    float* sp = stats + ((long long)b * 4 * K + 4 * k) * HW + pix;
    sp[0] = inv * invK;
    sp[HW] = f;
    sp[2 * HW] = mean;
    sp[3 * HW] = -sg * inv * invK + (float)ND * f * (xc - mean);
  }
}

// Image gradient, gathered at pixel q: d_x[k, q] = cen_k(q) + sum over (p, n) with clamp(p + o_n) = q of
//   da[p, n] A_k(p) sign(x_k(p) - x_k(q))   (|x_c - x_n| with x_n = x_k(q))
// + f_k(p) (x_k(q) - mean_k(p))            (the std sample x_k(q) of p)
__global__ void __launch_bounds__(256)
pamr_image_grad_kernel(const float* __restrict__ x, const float* __restrict__ da, int wpitch, const float* __restrict__ stats, int K,
                       int H, int W, Dil dil, float* __restrict__ dx) {
  const int px = blockIdx.x * kIterTW + (threadIdx.x % kIterTW);
  const int py = blockIdx.y * (256 / kIterTW) + (threadIdx.x / kIterTW);
  const int b = blockIdx.z;
  if (px >= W || py >= H) return;
  const long long HW = (long long)H * W, wplane = (long long)H * wpitch, q = (long long)py * W + px;
  const float* dab = da + (long long)b * 8 * dil.n * wplane;
  for (int k = 0; k < K; ++k) {
    const float* img = x + ((long long)b * K + k) * HW;
    const float* sp = stats + ((long long)b * 4 * K + 4 * k) * HW;
    const float xq = __ldg(img + q);
    float acc = __ldg(sp + 3 * HW + q);
    int n = 0;
    for (int di = 0; di < dil.n; ++di) {
      const int d = dil.d[di];
#pragma unroll
      for (int t = 0; t < 9; ++t) {
        if (t == 4) continue;
        int ylo, yhi, xlo, xhi;
        tap_sources(py, (t / 3 - 1) * d, H, ylo, yhi);
        tap_sources(px, (t % 3 - 1) * d, W, xlo, xhi);
        const float* dn = dab + n * wplane;
        for (int yy = ylo; yy <= yhi; ++yy)
          for (int xx = xlo; xx <= xhi; ++xx) {
            const long long p = (long long)yy * W + xx;
            const float u = __ldg(img + p) - xq;
            const float a = __ldg(dn + (long long)yy * wpitch + xx) * __ldg(sp + p);
            acc += u > 0.f ? a : (u < 0.f ? -a : 0.f);
            acc = fmaf(__ldg(sp + HW + p), xq - __ldg(sp + 2 * HW + p), acc);
          }
        ++n;
      }
    }
    dx[((long long)b * K + k) * HW + q] = acc;
  }
}

// Output rows (or columns) y in [0, n) whose bilinear taps may read source row i: y0(y) in {i - 1, i} needs
// i - 1 <= s * y < i + 1; one row of margin either side absorbs the rounding of fy = s * y.
__device__ __forceinline__ void up_sources(int i, float s, int n, int& lo, int& hi) {
  if (s <= 0.f) { lo = 0; hi = n - 1; return; }
  lo = (int)fmaxf(floorf((float)(i - 1) / s) - 1.f, 0.f);
  hi = (int)fminf(ceilf((float)(i + 1) / s) + 1.f, (float)(n - 1));
}

// Adjoint of pamr_upsample_kernel (unpadded): dmask[pl, i, j] = sum over output pixels (y, x) of the weight with which the
// forward's fp32 arithmetic read source pixel (i, j), times g[pl, y, x].  One thread per source pixel, any ratio.
__global__ void __launch_bounds__(256)
pamr_upsample_bwd_kernel(const float* __restrict__ g, int planes, int h, int w, int H, int W, float* __restrict__ dmask) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)planes * h * w) return;
  const int j = (int)(idx % w), i = (int)((idx / w) % h);
  const long long pl = idx / ((long long)h * w);
  const float sy = (H > 1) ? (float)(h - 1) / (float)(H - 1) : 0.f;
  const float sx = (W > 1) ? (float)(w - 1) / (float)(W - 1) : 0.f;
  int ylo, yhi, xlo, xhi;
  up_sources(i, sy, H, ylo, yhi);
  up_sources(j, sx, W, xlo, xhi);
  const float* gp = g + pl * H * W;
  float acc = 0.f;
  for (int y = ylo; y <= yhi; ++y) {
    const float fy = sy * (float)y;
    const int y0 = min((int)fy, h - 1), y1 = min(y0 + 1, h - 1);
    if (y0 != i && y1 != i) continue;
    const float ly = fy - (float)y0;
    const float cy = (y0 == i ? 1.f - ly : 0.f) + (y1 == i ? ly : 0.f);
    for (int x = xlo; x <= xhi; ++x) {
      const float fx = sx * (float)x;
      const int x0 = min((int)fx, w - 1), x1 = min(x0 + 1, w - 1);
      if (x0 != j && x1 != j) continue;
      const float lx = fx - (float)x0;
      const float cx = (x0 == j ? 1.f - lx : 0.f) + (x1 == j ? lx : 0.f);
      acc = fmaf(cy * cx, __ldg(gp + (long long)y * W + x), acc);
    }
  }
  dmask[idx] = acc;
}

template <template <int> class F, typename... A>
int by_nd(int nd, A... a) {
  switch (nd) {
    case 1: return F<1>::run(a...);
    case 2: return F<2>::run(a...);
    case 3: return F<3>::run(a...);
    case 4: return F<4>::run(a...);
    case 5: return F<5>::run(a...);
    case 6: return F<6>::run(a...);
    case 7: return F<7>::run(a...);
    default: return F<8>::run(a...);
  }
}

template <int ND>
struct WgradLaunch {
  static int run(const float* g, MaskBuf m, int B, int C, int H, int W, Dil dil, int first, float* dw, cudaStream_t st) {
    pamr_wgrad_kernel<ND><<<dim3((W + 127) / 128, H, B), 128, 0, st>>>(g, m, C, H, W, dil, wgt_pitch(W), first, dw);
    return acr::check_launch("pamr_wgrad_kernel");
  }
};

template <int ND>
struct AffinityBwdLaunch {
  static int run(const float* x, const float* wgt, int B, int K, int H, int W, Dil dil, float* dw, float* stats, cudaStream_t st) {
    pamr_affinity_bwd_kernel<ND><<<dim3((W + 127) / 128, H, B), 128, 0, st>>>(x, wgt, K, H, W, dil, wgt_pitch(W), dw, stats);
    return acr::check_launch("pamr_affinity_bwd_kernel");
  }
};

size_t grad_bytes(int B, int C, int H, int W) { return acr::align_up((size_t)B * C * H * W * sizeof(float), 256); }

int launch_upsample_bwd(const float* g, int planes, int mh, int mw, int H, int W, float* dmask, cudaStream_t st) {
  const long long total = (long long)planes * mh * mw;
  pamr_upsample_bwd_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(g, planes, mh, mw, H, W, dmask);
  return acr::check_launch("pamr_upsample_bwd_kernel");
}

// Argument checks shared by the entry points, in the order acr_pamr_fwd has always made them; fills `dil`.
int pamr_check(const char* fn, int B, int K, int C, int H, int W, int mh, int mw, const int* dilations_host, int nd, int num_iter,
               size_t ws_bytes, size_t ws_needed, Dil* dil) {
  ACR_REQUIRE(B > 0 && K > 0 && C > 0 && H > 0 && W > 0 && mh > 0 && mw > 0, ACR_E_INVAL, "%s: bad shape", fn);
  ACR_REQUIRE(nd >= 1 && nd <= kMaxDil, ACR_E_INVAL, "%s: 1 <= len(dilations) <= %d required", fn, kMaxDil);
  ACR_REQUIRE(num_iter >= 0, ACR_E_INVAL, "%s: num_iter < 0", fn);
  ACR_REQUIRE(ws_bytes >= ws_needed, ACR_E_NOMEM, "%s: workspace too small", fn);
  ACR_REQUIRE(H <= 65535 && (long long)B * C <= 65535, ACR_E_INVAL, "%s: grid too large", fn);
  dil->n = nd;
  for (int i = 0; i < kMaxDil; ++i) dil->d[i] = 0;
  for (int i = 0; i < nd; ++i) {
    ACR_REQUIRE(dilations_host[i] >= 1, ACR_E_INVAL, "%s: dilation < 1", fn);
    dil->d[i] = dilations_host[i];
  }
  return 0;
}

// The forward after its checks: up-sampling, weights, iterations (pamr_iterate's two buffer modes).
int pamr_run(const float* x, const float* mask, int B, int K, int C, int H, int W, int mh, int mw, const Dil& dil, int num_iter, float* out,
             float* wgt, float* ping, float* pong, size_t slot_stride, cudaStream_t st) {
  // the up-sampled mask goes to the padded ping buffer, or straight to `out` when there is nothing to iterate
  const int pad = num_iter > 0 ? kPamrHalo : 0;
  const long long total = (long long)B * C * (H + 2 * pad) * (W + 2 * pad);
  pamr_upsample_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(mask, B * C, mh, mw, H, W, pad, pad ? pad_pitch(W) : W,
                                                                        pad ? ping : out);
  if (int e = acr::check_launch("pamr_upsample_kernel")) return e;
  if (num_iter == 0) return 0;
  int e = 0;
  switch (dil.n) {
    case 1: e = launch_affinity_reg<1>(x, B, K, H, W, dil, wgt, st); break;
    case 2: e = launch_affinity_reg<2>(x, B, K, H, W, dil, wgt, st); break;
    case 3: e = launch_affinity_reg<3>(x, B, K, H, W, dil, wgt, st); break;
    case 4: e = launch_affinity_reg<4>(x, B, K, H, W, dil, wgt, st); break;
    case 5: e = launch_affinity_reg<5>(x, B, K, H, W, dil, wgt, st); break;
    case 6: e = launch_affinity_reg<6>(x, B, K, H, W, dil, wgt, st); break;
    case 7: e = launch_affinity_reg<7>(x, B, K, H, W, dil, wgt, st); break;
    default: e = launch_affinity_reg<8>(x, B, K, H, W, dil, wgt, st); break;
  }
  if (e) return e;
  return pamr_iterate(wgt, ping, pong, slot_stride, out, B, C, H, W, dil, num_iter, st);
}

}  // namespace

extern "C" size_t acr_pamr_workspace(int B, int K, int C, int H, int W, int nd) {
  if (B <= 0 || K <= 0 || C <= 0 || H <= 0 || W <= 0 || nd <= 0) return 0;
  return wgt_bytes(B, nd, H, W) + 2 * mask_bytes(B, C, H, W);
}

extern "C" int acr_pamr_fwd(const float* x, const float* mask, int B, int K, int C, int H, int W, int mh, int mw,
                            const int* dilations_host, int nd, int num_iter,
                            float* out, void* workspace, size_t workspace_bytes, void* stream) {
  ACR_REQUIRE(x && mask && out && workspace && dilations_host, ACR_E_INVAL, "acr_pamr_fwd: null pointer");
  Dil dil;
  if (int e = pamr_check("acr_pamr_fwd", B, K, C, H, W, mh, mw, dilations_host, nd, num_iter, workspace_bytes,
                         acr_pamr_workspace(B, K, C, H, W, nd), &dil))
    return e;
  float* wgt = (float*)workspace;
  float* ping = (float*)((char*)workspace + wgt_bytes(B, nd, H, W));
  float* pong = (float*)((char*)ping + mask_bytes(B, C, H, W));
  return pamr_run(x, mask, B, K, C, H, W, mh, mw, dil, num_iter, out, wgt, ping, pong, 0, (cudaStream_t)stream);
}

// saved = the weights, then one padded iterate M_t per slot (t = 0 .. num_iter - 1)
extern "C" size_t acr_pamr_save_workspace(int B, int K, int C, int H, int W, int nd, int num_iter) {
  if (B <= 0 || K <= 0 || C <= 0 || H <= 0 || W <= 0 || nd <= 0 || num_iter < 0) return 0;
  return wgt_bytes(B, nd, H, W) + (size_t)num_iter * mask_bytes(B, C, H, W);
}

extern "C" int acr_pamr_fwd_save(const float* x, const float* mask, int B, int K, int C, int H, int W, int mh, int mw,
                                 const int* dilations_host, int nd, int num_iter,
                                 float* out, void* saved, size_t saved_bytes, void* stream) {
  ACR_REQUIRE(x && mask && out && saved && dilations_host, ACR_E_INVAL, "acr_pamr_fwd_save: null pointer");
  Dil dil;
  if (int e = pamr_check("acr_pamr_fwd_save", B, K, C, H, W, mh, mw, dilations_host, nd, num_iter, saved_bytes,
                         acr_pamr_save_workspace(B, K, C, H, W, nd, num_iter), &dil))
    return e;
  float* slots = (float*)((char*)saved + wgt_bytes(B, nd, H, W));
  return pamr_run(x, mask, B, K, C, H, W, mh, mw, dil, num_iter, out, (float*)saved, slots, nullptr, mask_bytes(B, C, H, W),
                  (cudaStream_t)stream);
}

// two unpadded mask gradients (G_t ping-pong), the weight gradient / da planes, the 4K per-pixel factors of the image gradient
extern "C" size_t acr_pamr_bwd_workspace(int B, int K, int C, int H, int W, int nd) {
  if (B <= 0 || K <= 0 || C <= 0 || H <= 0 || W <= 0 || nd <= 0) return 0;
  return 2 * grad_bytes(B, C, H, W) + wgt_bytes(B, nd, H, W) + grad_bytes(B, 4 * K, H, W);
}

extern "C" int acr_pamr_bwd(const float* x, const void* saved, size_t saved_bytes, const float* g_out, int B, int K, int C, int H, int W,
                            int mh, int mw, const int* dilations_host, int nd, int num_iter, float* d_x, float* d_mask,
                            void* workspace, size_t workspace_bytes, void* stream) {
  ACR_REQUIRE(x && saved && g_out && workspace && dilations_host, ACR_E_INVAL, "acr_pamr_bwd: null pointer");
  ACR_REQUIRE(d_x || d_mask, ACR_E_INVAL, "acr_pamr_bwd: null pointer (neither d_x nor d_mask requested)");
  Dil dil;
  if (int e = pamr_check("acr_pamr_bwd", B, K, C, H, W, mh, mw, dilations_host, nd, num_iter, workspace_bytes,
                         acr_pamr_bwd_workspace(B, K, C, H, W, nd), &dil))
    return e;
  ACR_REQUIRE(saved_bytes >= acr_pamr_save_workspace(B, K, C, H, W, nd, num_iter), ACR_E_NOMEM, "acr_pamr_bwd: saved buffer too small");
  ACR_REQUIRE((long long)B * C * mh * mw <= 0x7fffffffLL && (long long)B * C * H * W <= 0x7fffffffLL, ACR_E_INVAL,
              "acr_pamr_bwd: grid too large");
  cudaStream_t st = (cudaStream_t)stream;
  const int T = num_iter;
  if (T == 0) {                                                    // out = up(mask): x does not reach the output
    if (d_x) ACR_CUDA(cudaMemsetAsync(d_x, 0, (size_t)B * K * H * W * sizeof(float), st));
    return d_mask ? launch_upsample_bwd(g_out, B * C, mh, mw, H, W, d_mask, st) : 0;
  }
  const float* wgt = (const float*)saved;
  auto iterate = [&](int t) { return padded_mask((float*)((char*)saved + wgt_bytes(B, nd, H, W) + (size_t)t * mask_bytes(B, C, H, W)), H, W); };
  float* gbuf[2] = {(float*)workspace, (float*)((char*)workspace + grad_bytes(B, C, H, W))};
  float* dw = (float*)((char*)workspace + 2 * grad_bytes(B, C, H, W));
  float* stats = (float*)((char*)dw + wgt_bytes(B, nd, H, W));
  const int groups = (C + kIterCG - 1) / kIterCG;
  const dim3 pix_grid((W + kIterTW - 1) / kIterTW, (H + 256 / kIterTW - 1) / (256 / kIterTW), B * groups);
  const float* g = g_out;                                          // G_t, from t = T down
  for (int t = T; t >= 1; --t) {
    if (d_x)
      if (int e = by_nd<WgradLaunch>(nd, g, iterate(t - 1), B, C, H, W, dil, (int)(t == T), dw, st)) return e;
    if (t == 1 && !d_mask) break;
    float* gn = gbuf[(T - t) & 1];
    pamr_iter_bwd_kernel<<<pix_grid, 256, 0, st>>>(wgt, wgt_pitch(W), g, gn, C, H, W, dil, groups);
    if (int e = acr::check_launch("pamr_iter_bwd_kernel")) return e;
    g = gn;
  }
  if (d_mask)
    if (int e = launch_upsample_bwd(g, B * C, mh, mw, H, W, d_mask, st)) return e;
  if (d_x) {
    if (int e = by_nd<AffinityBwdLaunch>(nd, x, wgt, B, K, H, W, dil, dw, stats, st)) return e;
    const dim3 img_grid(pix_grid.x, pix_grid.y, B);
    pamr_image_grad_kernel<<<img_grid, 256, 0, st>>>(x, dw, wgt_pitch(W), stats, K, H, W, dil, d_x);
    if (int e = acr::check_launch("pamr_image_grad_kernel")) return e;
  }
  return 0;
}
