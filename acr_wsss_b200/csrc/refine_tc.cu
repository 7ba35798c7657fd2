// (a9) on the tensor cores: the two dense contractions of CAM generation,
//   patch CAM   relu(cls_head(layer4[:,1:]))            DPT/ACR.py:133-134   [Np x E] x [E x C]
//   refinement  (sum_l attn[:,l,1:,1:])^t . cam          infer_cam.py:164-165,184   [Np x Np] x [Np x C']
// as ONE kernel: a "tall-skinny" fp32 contraction out[M x Nc] = (sum over L slabs of A)[M x K] . Bm[K x Nc], Nc <= 128.
//
// Both are HBM-bound streams of the A operand (the refinement reads L*Np*Np*4 bytes = 29.5 MB per view at 448x448 to
// produce Np*C' numbers), so the kernel is built around that stream:
//   * the L head-mean maps are summed in registers while they are read (the [B,Np,Np] matrix A is never materialised
//     for t = 1; for t > 1 the first pass also writes it once and the later powers re-read 2.46 MB instead of 29.5 MB),
//   * the products run on tcgen05 with the fp32 operands split into bf16 hi + lo parts in shared memory
//     (hi.hi + lo.hi + hi.lo, fp32 accumulation in TMEM: relative error ~2^-16, inside the fp32 parity budget of 1e-3;
//     a plain bf16 or tf32 product is not),
//   * K is split over a thread-block CLUSTER (up to 8 CTAs) so that 7 row tiles x 2 views still fill the GPU; the
//     partial [128 x Nc] tiles are reduced through distributed shared memory in rank order (deterministic),
//   * row normalisation (A / rowsum(A)) is an extra all-ones column of Bm: the row sums come out of the same MMAs and
//     the division happens in the epilogue, as do the bias and the relu of the patch-CAM head.
#include "attn_tc.cuh"
#include <cooperative_groups.h>

namespace cg = cooperative_groups;

namespace {

constexpr int TM = 128;              // output rows per CTA (UMMA M)
constexpr int TK = 64;               // K per stage: one 128-byte SWIZZLE_128B row of bf16
constexpr int NC_MAX = 128;          // padded output columns (UMMA N), multiple of 32
constexpr int THREADS = 512;         // 16 warps x 8 rows of the A tile
constexpr uint32_t A_BYTES = TM * TK * 2;      // 16 KB: a [128 x 64] bf16 operand tile

// Dynamic shared memory (1024-byte aligned): two operand stages {A hi, A lo, B hi, B lo} with B tiles of ncp rows,
// aliased after the last MMA by this CTA's fp32 partial tile [128][ncp + 1]; then the row sums, barriers, TMEM base.
struct Tail {
  float rowsum[TM];
  uint64_t mma_done[2];
  uint32_t tmem_base;
};
__host__ __device__ inline uint32_t stage_bytes(int ncp) { return 2 * A_BYTES + 2 * (uint32_t)ncp * TK * 2; }
__host__ __device__ inline uint32_t ring_bytes(int ncp) {
  const uint32_t ring = 2 * stage_bytes(ncp), part = (uint32_t)(TM * (ncp + 1) * sizeof(float));
  return ((ring > part ? ring : part) + 1023u) & ~1023u;
}

struct Params {
  const float* A; long long a_bs, a_ls, a_rs; int L, M, K;      // A[b,l,i,k] = A[b*a_bs + l*a_ls + i*a_rs + k]
  const float* Bm; long long b_bs, b_ks, b_ns; int Nc, ncp;     // Bm[b,k,n] = Bm[b*b_bs + k*b_ks + n*b_ns]; ncp = padded columns
  float* out; long long o_bs, o_rs;                             // out[b,i,n]
  float* a_out;                                                 // optional dense [B,M,K]: the slab sum of A
  const float* bias; int relu, normalize;
};

// byte offset of element (row r, column k) of a K-major [rows x 64] bf16 tile in SWIZZLE_128B layout
__device__ __forceinline__ uint32_t sw128(int r, int k) {
  return (uint32_t)((r >> 3) * 1024 + (r & 7) * 128 + ((((k >> 3) ^ (r & 7)) << 4) | ((k & 7) << 1)));
}
__device__ __forceinline__ void split_store(uint8_t* hi_tile, uint8_t* lo_tile, uint32_t off, float v) {
  const __nv_bfloat16 h = __float2bfloat16_rn(v);
  const __nv_bfloat16 l = __float2bfloat16_rn(v - __bfloat162float(h));
  *reinterpret_cast<__nv_bfloat16*>(hi_tile + off) = h;
  *reinterpret_cast<__nv_bfloat16*>(lo_tile + off) = l;
}

__global__ void __launch_bounds__(THREADS, 1) refine_tc_kernel(const Params p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* ring = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int ncp = p.ncp, LDP = ncp + 1;
  float* part = reinterpret_cast<float*>(ring);
  Tail& s = *reinterpret_cast<Tail*>(ring + ring_bytes(ncp));
  const uint32_t sbytes = stage_bytes(ncp), b_bytes = (uint32_t)ncp * TK * 2;
  cg::cluster_group cluster = cg::this_cluster();
  const int ks = (int)cluster.num_blocks(), rank = (int)cluster.block_rank();     // cluster = K split, along grid x
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m0 = blockIdx.y * TM, b = blockIdx.z;
  const int nchunks = (p.K + TK - 1) / TK;
  const int c_begin = (int)((long long)nchunks * rank / ks), c_end = (int)((long long)nchunks * (rank + 1) / ks);

  if (threadIdx.x == 0) {
    tc::mbar_init(&s.mma_done[0], 1);
    tc::mbar_init(&s.mma_done[1], 1);
    tc::fence_barrier_init();
  }
  if (warp == 0) tc::tmem_alloc<NC_MAX>(&s.tmem_base);
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tD = s.tmem_base;
  const uint32_t idesc = tc::idesc_bf16_f32(TM, ncp, 0, 0);

  const float* Ab = p.A + (long long)b * p.a_bs;
  const float* Bb = p.Bm + (long long)b * p.b_bs;
  // L == 1 (patch CAM, later powers of A): the 16 values of a thread's share of chunk c + 1 are in flight while chunk c is
  // converted, published and multiplied.  L > 1: 8 rows x 2 columns x 4 slabs = 64 independent loads per round trip.
  float x1[8][2];
  auto load_l1 = [&](int c) {
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int row = m0 + warp * 8 + u;
#pragma unroll
      for (int v = 0; v < 2; ++v) {
        const int k = c * TK + lane + 32 * v;
        x1[u][v] = (c < c_end && row < p.M && k < p.K) ? __ldg(Ab + (long long)row * p.a_rs + k) : 0.f;
      }
    }
  };
  if (p.L == 1) load_l1(c_begin);
  for (int c = c_begin; c < c_end; ++c) {
    const int i = c - c_begin, sidx = i & 1, k0 = c * TK;
    uint8_t* a_hi = ring + sidx * sbytes, *a_lo = a_hi + A_BYTES, *b_hi = a_lo + A_BYTES, *b_lo = b_hi + b_bytes;
    if (i >= 2) tc::mbar_wait(&s.mma_done[sidx], ((i >> 1) - 1) & 1);      // the MMAs that read this stage have retired
    if (p.L == 1) {
#pragma unroll
      for (int u = 0; u < 8; ++u)
#pragma unroll
        for (int v = 0; v < 2; ++v) split_store(a_hi, a_lo, sw128(warp * 8 + u, lane + 32 * v), x1[u][v]);
      load_l1(c + 1);
    } else {
      const int r = warp * 8;
      float acc[8][2];
      bool ok[8][2];
      int off[8][2];
#pragma unroll
      for (int u = 0; u < 8; ++u)
#pragma unroll
        for (int v = 0; v < 2; ++v) {
          acc[u][v] = 0.f;
          ok[u][v] = m0 + r + u < p.M && k0 + lane + 32 * v < p.K;
          off[u][v] = ok[u][v] ? (int)((m0 + r + u) * p.a_rs + k0 + lane + 32 * v) : 0;
        }
#pragma unroll 4
      for (int l = 0; l < p.L; ++l) {
        const float* slab = Ab + (long long)l * p.a_ls;
#pragma unroll
        for (int u = 0; u < 8; ++u)
#pragma unroll
          for (int v = 0; v < 2; ++v) acc[u][v] += __ldg(slab + off[u][v]);
      }
#pragma unroll
      for (int u = 0; u < 8; ++u)
#pragma unroll
        for (int v = 0; v < 2; ++v) {
          const float x = ok[u][v] ? acc[u][v] : 0.f;
          if (p.a_out != nullptr && ok[u][v]) p.a_out[((long long)b * p.M + m0 + r + u) * p.K + k0 + lane + 32 * v] = x;
          split_store(a_hi, a_lo, sw128(r + u, lane + 32 * v), x);
        }
    }
    // ---- Bm chunk [64 k x ncp n] -> K-major tile [n][k]; column Nc is the all-ones column when normalising
    for (int idx = threadIdx.x; idx < TK * ncp; idx += THREADS) {
      int k, n;
      if (p.b_ks == 1) { k = idx & (TK - 1); n = idx >> 6; } else { n = idx % ncp; k = idx / ncp; }
      const int kk = k0 + k;
      float x = 0.f;
      if (kk < p.K) {
        if (n < p.Nc) x = __ldg(Bb + (long long)kk * p.b_ks + (long long)n * p.b_ns);
        else if (n == p.Nc && p.normalize) x = 1.f;
      }
      split_store(b_hi, b_lo, sw128(n, k), x);
    }
    tc::fence_proxy_async_smem();
    __syncthreads();
    if (warp == 0) {
      tc::tc_fence_after();
      const uint64_t dah = tc::smem_desc_sw128(tc::smem_u32(a_hi), 16, 1024), dal = tc::smem_desc_sw128(tc::smem_u32(a_lo), 16, 1024);
      const uint64_t dbh = tc::smem_desc_sw128(tc::smem_u32(b_hi), 16, 1024), dbl = tc::smem_desc_sw128(tc::smem_u32(b_lo), 16, 1024);
      if (tc::elect_one()) {
#pragma unroll
        for (int q = 0; q < TK / 16; ++q) {
          tc::mma_ss_off(tD, dah, q * 2, dbh, q * 2, idesc, (i > 0) || (q > 0));
          tc::mma_ss_off(tD, dal, q * 2, dbh, q * 2, idesc, 1);
          tc::mma_ss_off(tD, dah, q * 2, dbl, q * 2, idesc, 1);
        }
        tc::tc_commit(&s.mma_done[sidx]);
      }
      __syncwarp();
    }
  }
  // ---- this CTA's partial tile: TMEM -> registers -> shared memory (the operand ring is free once the last MMA retired)
  const int nloc = c_end - c_begin;
  if (nloc > 0) {
    tc::mbar_wait(&s.mma_done[(nloc - 1) & 1], ((nloc - 1) >> 1) & 1);
    tc::tc_fence_after();
  }
  __syncthreads();
  {
    const int quad = warp & 3;                                  // TMEM lane quadrant of this warp
    const int row = quad * 32 + lane;
    for (int cch = warp >> 2; cch * 32 < ncp; cch += THREADS / 128) {      // 32-column chunks
      uint32_t r[32];
      if (nloc > 0) {
        tc::tmem_ld32(tD + ((uint32_t)(quad * 32) << 16) + cch * 32, r);
        tc::tmem_ld_wait();
      } else {
#pragma unroll
        for (int e = 0; e < 32; ++e) r[e] = 0u;
      }
#pragma unroll
      for (int e = 0; e < 32; ++e) part[row * LDP + cch * 32 + e] = __uint_as_float(r[e]);
    }
  }
  tc::tc_fence_before();
  cluster.sync();
  // ---- reduce over the K split through distributed shared memory (rank order), epilogue, store
  const int rows_per = TM / ks, r0 = rank * rows_per;
  if (p.normalize) {
    for (int t = threadIdx.x; t < rows_per; t += THREADS) {
      float v = 0.f;
      for (int q = 0; q < ks; ++q) v += cluster.map_shared_rank(part, q)[(r0 + t) * LDP + p.Nc];
      s.rowsum[t] = v;
    }
    __syncthreads();
  }
  for (int idx = threadIdx.x; idx < rows_per * p.Nc; idx += THREADS) {
    const int rl = idx / p.Nc, col = idx - rl * p.Nc;
    const int row = m0 + r0 + rl;
    if (row >= p.M) break;
    float v = 0.f;
    for (int q = 0; q < ks; ++q) v += cluster.map_shared_rank(part, q)[(r0 + rl) * LDP + col];
    if (p.normalize) v /= s.rowsum[rl];
    if (p.bias != nullptr) v += __ldg(p.bias + col);
    if (p.relu) v = fmaxf(v, 0.f);
    p.out[(long long)b * p.o_bs + (long long)row * p.o_rs + col] = v;
  }
  cluster.sync();                                            // nobody leaves while its tile is still being read
  if (warp == 0) {
    tc::tc_fence_after();
    tc::tmem_dealloc<NC_MAX>(tD);
  }
}

int launch_refine(const Params& p, int B, const char* what, cudaStream_t st) {
  const int mt = (p.M + TM - 1) / TM, nchunks = (p.K + TK - 1) / TK;
  // K split (cluster size): fewest (waves of CTAs) x (chunks per CTA), one CTA per SM
  int ks = 1;
  long long best = -1;
  for (int c = 1; c <= 8 && c <= nchunks; c *= 2) {
    const long long cost = (((long long)mt * B * c + 147) / 148) * ((nchunks + c - 1) / c);
    if (best < 0 || cost < best) { best = cost; ks = c; }
  }
  const size_t smem = ring_bytes(p.ncp) + sizeof(Tail) + 1024;
  static bool attr_set[64] = {false};
  if (int e = acr_attn::set_max_smem(refine_tc_kernel, ring_bytes(NC_MAX) + sizeof(Tail) + 1024, attr_set)) return e;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(ks, mt, B);
  cfg.blockDim = dim3(THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = ks;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  acr::KernelTimer kt_(what, st);
  ACR_CUDA(cudaLaunchKernelEx(&cfg, refine_tc_kernel, p));
  return acr::check_launch(what);
}

int padded_cols(int n) { return (n + 31) / 32 * 32; }

}  // namespace

extern "C" size_t acr_affinity_refine_tc_workspace(int B, int N, int C, int t) {
  if (B <= 0 || N <= 1 || C <= 0 || t <= 1) return 0;
  const size_t Np = (size_t)N - 1;
  return acr::align_up((size_t)B * Np * Np * sizeof(float), 256) + acr::align_up((size_t)B * Np * C * sizeof(float), 256);
}

extern "C" int acr_affinity_refine_tc(const float* attn, int B, int L, int N, const float* cam, int C, int t, int normalize,
                                      float* out, void* workspace, size_t workspace_bytes, void* stream) {
  ACR_REQUIRE(attn && cam && out, ACR_E_INVAL, "acr_affinity_refine_tc: null pointer");
  ACR_REQUIRE(B > 0 && B <= 65535 && L > 0 && N > 1 && C > 0 && t >= 1, ACR_E_INVAL, "acr_affinity_refine_tc: bad shape");
  ACR_REQUIRE(C + (normalize ? 1 : 0) <= NC_MAX, ACR_E_INVAL, "acr_affinity_refine_tc: C + normalize must be <= %d (C = %d, normalize = %d)",
              NC_MAX, C, normalize ? 1 : 0);
  ACR_REQUIRE(t == 1 || (workspace && ((uintptr_t)workspace & 255) == 0 && workspace_bytes >= acr_affinity_refine_tc_workspace(B, N, C, t)),
              ACR_E_NOMEM, "acr_affinity_refine_tc: t > 1 needs acr_affinity_refine_tc_workspace() bytes, 256-byte aligned");
  ACR_REQUIRE(acr_device_is_sm100(), ACR_E_NOSM100, "acr_affinity_refine_tc: needs an sm_100 device");
  const int Np = N - 1;
  float* wsA = t > 1 ? (float*)workspace : nullptr;
  float* tmp = t > 1 ? (float*)((char*)workspace + acr::align_up((size_t)B * Np * Np * sizeof(float), 256)) : nullptr;
  const float* src = cam;
  for (int sidx = 0; sidx < t; ++sidx) {
    float* dst = ((t - 1 - sidx) % 2 == 0) ? out : tmp;      // ping-pong so that the t-th product lands in `out`
    Params p = {};
    if (sidx == 0) {                                         // patch x patch part of the maps, summed over the L blocks on the fly
      p.A = attn + (long long)N + 1; p.a_bs = (long long)L * N * N; p.a_ls = (long long)N * N; p.a_rs = N; p.L = L;
      p.a_out = wsA;
    } else {
      p.A = wsA; p.a_bs = (long long)Np * Np; p.a_ls = 0; p.a_rs = Np; p.L = 1;
    }
    p.M = Np; p.K = Np;
    p.Bm = src; p.b_bs = (long long)Np * C; p.b_ks = C; p.b_ns = 1; p.Nc = C; p.ncp = padded_cols(C + (normalize ? 1 : 0));
    p.out = dst; p.o_bs = (long long)Np * C; p.o_rs = C;
    p.normalize = normalize ? 1 : 0;
    if (int e = launch_refine(p, B, "affinity_refine_tc", (cudaStream_t)stream)) return e;
    src = dst;
  }
  return 0;
}

extern "C" int acr_patch_cam_tc(const float* tokens, long long tok_batch_stride, long long tok_row_stride, int B, int M, int E,
                                const float* weight, const float* bias, int C, int relu, float* out, void* stream) {
  ACR_REQUIRE(tokens && weight && out, ACR_E_INVAL, "acr_patch_cam_tc: null pointer");
  ACR_REQUIRE(B > 0 && B <= 65535 && M > 0 && E > 0 && C > 0 && C <= NC_MAX, ACR_E_INVAL, "acr_patch_cam_tc: bad shape (C <= %d)", NC_MAX);
  ACR_REQUIRE(tok_row_stride >= E, ACR_E_INVAL, "acr_patch_cam_tc: token row stride < E");
  ACR_REQUIRE(acr_device_is_sm100(), ACR_E_NOSM100, "acr_patch_cam_tc: needs an sm_100 device");
  Params p = {};
  p.A = tokens; p.a_bs = tok_batch_stride; p.a_ls = 0; p.a_rs = tok_row_stride; p.L = 1; p.M = M; p.K = E;
  p.Bm = weight; p.b_bs = 0; p.b_ks = 1; p.b_ns = E; p.Nc = C; p.ncp = padded_cols(C);       // nn.Linear weight [C,E]: K-major as stored
  p.out = out; p.o_bs = (long long)M * C; p.o_rs = C;
  p.bias = bias; p.relu = relu ? 1 : 0;
  return launch_refine(p, B, "patch_cam_tc", (cudaStream_t)stream);
}
