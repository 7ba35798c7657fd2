// (a1, backward) Fused attention backward for sm_100a.  models/vision_transformer.py:203-211 differentiated, plus the
// dense additive term the head-mean affinity (DPT/ACR.py:107-112) sends back into every head:
//   dP_h = dO_h V_h^T + G/H ;  dS_h = P_h * (dP_h - delta) ;  dV = P^T dO ; dK = dS^T Q * scale ; dQ = dS K * scale
// (delta comes from bwd_delta_kernel + attn_mean_kernel<1>, attn_tc.cu).
//
// Work item = (key tile j, head, image): K_j, V_j stationary, loop over query tiles i; a persistent grid of one CTA per SM
// walks over the items.  512 threads, five roles:
//   warp 0      TMA producer: K, V once per item; per query tile Q_i, dO_i (three-stage ring running across items)
//   warp 1      MMA issuer (one thread): S = Q_i K_j^T, dP = dO_i V_j^T (SS, 128x128x64), then dV += P^T dO_i,
//               dK += dS^T Q_i, dQ_i = dS K_j from the bf16 P / dS tiles the softmax warps publish in shared memory
//   warps 2-3   row statistics (log2-domain LSE, delta) of the next query tile into shared memory
//   warps 4-11  softmax backward: a thread owns one query row x 64 key columns.  It pulls S and dP out of TMEM into
//               registers in one go and hands tS/tDP back at once (sdp_free), so the scores of tile i+1 run on the tensor
//               pipe UNDER the exponentials of tile i; P and dS stay in registers until the gradient MMAs of tile i-1 have
//               released the single-buffered smem tiles (pds_free)
//   warps 12-15 drain: per tile dQ from TMEM -> 64-bit fixed-point staging -> four cp.reduce.async.bulk.tensor (u64 add,
//               order-independent, so the result is the same every run); per item
//               dK / dV from TMEM -> bf16 rows of d_qkv
// The softmax warps therefore execute nothing but the element-wise chain (round 1's kernel spent ~75 % of their time in
// barrier waits, the dQ hand-over and the exposed S/dP MMA latency: profiles/r01g_ncu_attn_bwd_full.txt).
// Element-wise math uses the packed fp32x2 instructions (FFMA2 / FMUL2 / FADD2): 5 issue slots per element instead of 8.
#include "attn_tc.cuh"

using namespace acr_attn;

namespace {

constexpr int NST = 3;

struct BwdSmem {
  uint8_t k[TILE_BYTES];
  uint8_t v[TILE_BYTES];
  uint8_t q[NST][TILE_BYTES];      // Q_i / dO_i ring: three stages, because a slot is only released by the gradient MMAs of its
  uint8_t d_o[NST][TILE_BYTES];    // tile and the TMA refill takes ~1500 cycles (two stages left that latency exposed every tile)
  uint8_t p[2][TILE_BYTES];        // [kv block of 64][q row][64 kv] bf16, SWIZZLE_128B rows (one row per thread)
  uint8_t ds[2][TILE_BYTES];       // same layout: read MN-major (A = dS^T / P^T) and K-major (A = dS)
  uint8_t dq[2][TILE_BYTES];       // dQ staging: two [q row][16 u64 fixed-point columns] boxes, SWIZZLE_128B (see drain_box)
  float stat[2][2][BM];            // [tile parity][0: lse * log2(e), 1: delta][q row]
  uint64_t kv_full, kv_empty, dkv_free, qdo_full[NST], qdo_empty[NST], stat_full[2], sdp_full, sdp_free, pds_full, pds_free, dq_full, dq_free;
  uint32_t tmem_base;
};
static_assert(sizeof(BwdSmem) <= 232448, "BwdSmem exceeds the 227 KB dynamic shared memory limit");

constexpr int BWD_THREADS = 512;

// clock64 timeline of one CTA (development builds only: scripts/micro/bwd_trace.cu compiles this file with -DACR_BWD_TRACE)
#ifdef ACR_BWD_TRACE
__device__ unsigned long long g_bwd_trace[4][16][8];      // [role][tile][event]
#define BWD_TRACE(role, tile, ev)                                                                         \
  do {                                                                                                    \
    if (blockIdx.x == 5 && (tile) < 16 && (threadIdx.x & 31) == 0) g_bwd_trace[role][tile][ev] = clock64(); \
  } while (0)
#else
#define BWD_TRACE(role, tile, ev) do { } while (0)
#endif
constexpr int REG_CTRL = 48, REG_DRAIN = 64, REG_SOFTMAX = 200;      // 128*48 + 128*64 + 256*200 = 65536

// ---- packed fp32x2 arithmetic (sm_100: one issue slot for two lanes of fp32 math)
__device__ __forceinline__ uint64_t f2_pack(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void f2_unpack(uint64_t v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ uint64_t f2_fma(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ uint64_t f2_mul(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ uint64_t f2_add(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
// Softmax backward of one thread's share of a tile: query row `row`, key columns colbase .. colbase+63 (`half` of the tile).
// Pulls S / dP out of TMEM 32 columns at a time, releases them (sdp_free) after the second pull and writes P and dS as bf16
// into this thread's rows of the swizzled shared-memory tiles (p_row / ds_row: shared addresses of the row start).  The tiles are
// single-buffered: the first store waits for the gradient MMAs of the previous tile (pds_free, parity pds_par; < 0: no wait).
// GMODE: 0 no affinity gradient, 1 fp32 rows (scalar loads, bounds checked), 2 fp32 rows (128-bit loads), 3 sign codes
// (64 bytes of this row in cwt, loaded one tile ahead; `gw` then carries 2*w*scale/H of this row, otherwise 1/H).
template <int GMODE, bool TAIL>
__device__ __forceinline__ void bwd_softmax_tile(BwdSmem& s, uint32_t tS, uint32_t tDP, uint32_t tDS, uint32_t lane_off, int half, int row, int colbase, int N,
                                                 const float* __restrict__ grow, const uint32_t (&cwt)[16], float gw, float scale_log2, float lse2,
                                                 float dlt, float* __restrict__ rd_row0, uint32_t p_row, uint32_t ds_row, int pds_par) {
  const int nlive = TAIL ? (N - colbase) : 64;         // live key columns of this thread (warp-uniform; may be <= 0)
  const uint64_t sc2 = f2_pack(scale_log2, scale_log2), nl2 = f2_pack(-lse2, -lse2), nd2 = f2_pack(-dlt, -dlt), gw2 = f2_pack(gw, gw);
  uint32_t pk[32], dk[32];        // P and dS of the whole tile as packed bf16 pairs: held until the previous tile's gradient MMAs retire
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    // 32 columns at a time (a tcgen05.ld.x32 needs 32 consecutive registers; four such blocks live at once made ptxas spill)
    uint32_t rs[32], rd[32];
    const bool live = !TAIL || c * 32 < nlive;
    if (live) {
      tc::tmem_ld32(tS + lane_off + half * 64 + c * 32, rs);
      tc::tmem_ld32(tDP + lane_off + half * 64 + c * 32, rd);
      tc::tmem_ld_wait();
    }
    if (c == 1) {
      // tS / tDP may be overwritten by the scores of the next tile.  Half-way through the body is early enough: the tensor
      // pipe is busy with the gradient MMAs of the previous tile until then anyway.
      tc::tc_fence_before();
      tc::mbar_arrive(&s.sdp_free);
      if (half == 0 && row < 32) BWD_TRACE(1, 15, 2);
    }
    if (!live) {
#pragma unroll
      for (int e = 0; e < 16; ++e) pk[c * 16 + e] = dk[c * 16 + e] = 0u;
    } else {
    const uint32_t* cw = cwt + c * 8;        // sign codes of these 32 columns (GMODE 3), prefetched by the caller
    float g[GMODE == 1 || GMODE == 2 ? 32 : 1];
    if (GMODE == 2) {
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(grow + c * 32) + e);
        g[4 * e] = t.x; g[4 * e + 1] = t.y; g[4 * e + 2] = t.z; g[4 * e + 3] = t.w;
      }
    } else if (GMODE == 1) {
#pragma unroll
      for (int e = 0; e < 32; ++e) g[e] = (colbase + c * 32 + e < N) ? __ldg(grow + c * 32 + e) : 0.f;
    }
    if (rd_row0 != nullptr) {        // row 0 of dP_h incl. the affinity term (one thread of one tile): what the reference's hook keeps
#pragma unroll
      for (int e = 0; e < 32; ++e) {
        float gv = 0.f;
        if (GMODE == 3) gv = __uint_as_float((((cw[e >> 2] >> ((e & 3) * 8)) & 0xffu) << 24));
        else if (GMODE != 0) gv = g[e];
        if (colbase + c * 32 + e < N) rd_row0[c * 32 + e] = fmaf(gv, gw, __uint_as_float(rd[e]));
      }
    }
#pragma unroll
    for (int e = 0; e < 16; ++e) {
      const int i0 = c * 32 + 2 * e;
      const uint64_t x = f2_fma(f2_pack(__uint_as_float(rs[2 * e]), __uint_as_float(rs[2 * e + 1])), sc2, nl2);
      float x0, x1;
      f2_unpack(x, x0, x1);
      float p0 = tc::fast_exp2(x0), p1 = tc::fast_exp2(x1);
      if (TAIL) {
        if (i0 >= nlive) p0 = 0.f;
        if (i0 + 1 >= nlive) p1 = 0.f;
      }
      uint64_t dp = f2_pack(__uint_as_float(rd[2 * e]), __uint_as_float(rd[2 * e + 1]));
      if (GMODE == 3) {
        float g0 = ACR_CODE_F(cw[e >> 1], (2 * e) & 3), g1 = ACR_CODE_F(cw[e >> 1], (2 * e + 1) & 3);
        if (TAIL) {        // bytes past N are row padding: whatever they hold is no gradient
          if (i0 >= nlive) g0 = 0.f;
          if (i0 + 1 >= nlive) g1 = 0.f;
        }
        dp = f2_fma(f2_pack(g0, g1), gw2, dp);
      } else if (GMODE != 0) {
        dp = f2_fma(f2_pack(g[2 * e], g[2 * e + 1]), gw2, dp);
      }
      const uint64_t dsv = f2_mul(f2_pack(p0, p1), f2_add(dp, nd2));
      float d0, d1;
      f2_unpack(dsv, d0, d1);
      pk[c * 16 + e] = tc::pack_bf16(p0, p1);
      dk[c * 16 + e] = tc::pack_bf16(d0, d1);
    }
    }   // live
  }
  // The P / dS tiles are single-buffered: the dV / dK MMAs of the previous tile (pds_free) and its dQ MMA (dq_full, reads tDS)
  // must have retired.  Waiting here, after the whole tile has been computed, keeps that off the critical path.
  if (pds_par >= 0) {
    if (half == 0 && row < 32) BWD_TRACE(1, 15, 3);
    tc::mbar_wait(&s.pds_free, (uint32_t)pds_par);
    tc::mbar_wait(&s.dq_full, (uint32_t)pds_par);
    tc::tc_fence_after();
    if (half == 0 && row < 32) BWD_TRACE(1, 15, 5);
  }
#pragma unroll
  for (int cc = 0; cc < 8; ++cc) {               // 16-byte chunk cc of this row at position cc ^ (row & 7)
    // p_row / ds_row = (row start) ^ ((row & 7) << 4): rows are 128-byte aligned, so one XOR with an immediate addresses the chunk
    sts128(p_row ^ (uint32_t)(cc << 4), pk[cc * 4 + 0], pk[cc * 4 + 1], pk[cc * 4 + 2], pk[cc * 4 + 3]);
    sts128(ds_row ^ (uint32_t)(cc << 4), dk[cc * 4 + 0], dk[cc * 4 + 1], dk[cc * 4 + 2], dk[cc * 4 + 3]);
  }
  // dS a second time, as the TMEM-resident A operand of dQ = dS K (64 keys = 32 packed columns): the dQ MMA then reads only K
  // from shared memory, whose bandwidth (128 B/clk) is what bounds this kernel
  tc::tmem_st16(tDS + lane_off + half * 32, dk);
  tc::tmem_st16(tDS + lane_off + half * 32 + 16, dk + 16);
  tc::tmem_st_wait();
}

struct SoftmaxArgs {
  uint32_t tS, tDP, tDS, lane_off;
  int half, row, colbase, N, H, ntiles, b, h;
  const float* g_mean;
  long long g_bs, g_ld;
  float* g_row0;
  const unsigned char* code;
  long long code_bs, code_ld;
  float w_cls2, w_aff2, invH, scale_log2;
  uint32_t p_row, ds_row, swz;
};

// The query-tile loop of one softmax thread for one work item; T0 = tiles this CTA has processed before it (the mbarrier
// parities run on the CTA-wide tile count).
template <int GMODE, bool TAIL>
__device__ __forceinline__ void bwd_softmax_loop(BwdSmem& s, const SoftmaxArgs& a, int T0) {
  const int row = a.row, N = a.N;
  const int wq = row & ~31;                            // first row of this warp's TMEM lane quadrant
  // Sign codes: 64 bytes of this thread's row per tile, straight from global memory (each byte is used by one thread of one
  // CTA per head, so staging through shared memory would only add traffic to the resource that bounds the kernel); the loads
  // of tile i+1 are issued at the top of tile i.  Rows past N read the (valid) last row: their P is 0.
  uint32_t cwn[16];
  auto load_codes = [&](int i) {
    const uint4* src = reinterpret_cast<const uint4*>(a.code + (size_t)a.b * a.code_bs + (size_t)min(i * BM + row, N - 1) * a.code_ld + a.colbase);
#pragma unroll
    for (int v = 0; v < 4; ++v) {
      uint4 t = make_uint4(0u, 0u, 0u, 0u);
      if (!TAIL || a.colbase + v * 16 < N) t = __ldg(src + v);
      cwn[v * 4 + 0] = t.x; cwn[v * 4 + 1] = t.y; cwn[v * 4 + 2] = t.z; cwn[v * 4 + 3] = t.w;
    }
  };
  if (GMODE == 3) load_codes(0);
  for (int i = 0; i < a.ntiles; ++i) {
    uint32_t cw[16];
    if (GMODE == 3) {
#pragma unroll
      for (int v = 0; v < 16; ++v) cw[v] = cwn[v];
      if (i + 1 < a.ntiles) load_codes(i + 1);
    }
    const int q0 = i * BM;
    const int T = T0 + i;
    const int pds_par = (T > 0) ? ((T - 1) & 1) : -1;
    const int qi = q0 + row;
    const bool rows_live = q0 + wq < N;                // warp-uniform
    float lse2 = INFINITY, dlt = 0.f;
    if (rows_live) {
      tc::mbar_wait(&s.stat_full[T & 1], (T >> 1) & 1);
      lse2 = s.stat[T & 1][0][row];
      dlt = s.stat[T & 1][1][row];
    }
    if (a.half == 0 && row < 32) BWD_TRACE(1, i, 0);
    tc::mbar_wait(&s.sdp_full, T & 1);
    tc::tc_fence_after();
    if (a.half == 0 && row < 32) BWD_TRACE(1, i, 1);
    if (!rows_live) {
      // all 32 query rows of this warp lie past N (last query tile): the tiles just need finite values there (they meet
      // zero-filled dO / Q rows in the gradient MMAs)
      tc::tc_fence_before();
      tc::mbar_arrive(&s.sdp_free);
      if (pds_par >= 0) {
        tc::mbar_wait(&s.pds_free, (uint32_t)pds_par);
        tc::mbar_wait(&s.dq_full, (uint32_t)pds_par);
        tc::tc_fence_after();
      }
#pragma unroll
      for (int cc = 0; cc < 8; ++cc) {
        sts128(a.p_row ^ (uint32_t)(cc << 4), 0u, 0u, 0u, 0u);
        sts128(a.ds_row ^ (uint32_t)(cc << 4), 0u, 0u, 0u, 0u);
      }
      {
        uint32_t z[16];
#pragma unroll
        for (int e = 0; e < 16; ++e) z[e] = 0u;
        tc::tmem_st16(a.tDS + a.lane_off + a.half * 32, z);
        tc::tmem_st16(a.tDS + a.lane_off + a.half * 32 + 16, z);
        tc::tmem_st_wait();
      }
    } else {
      // rows past N inside a live warp read a clamped (valid) row of G: their P is 0, so the value is irrelevant (the tile body
      // contains warp-collective tcgen05.ld, so all lanes run it)
      const float* grow = (GMODE == 1 || GMODE == 2) ? a.g_mean + (size_t)a.b * a.g_bs + (size_t)min(qi, N - 1) * a.g_ld + a.colbase : nullptr;
      float* rd_row0 = (a.g_row0 != nullptr && qi == 0) ? a.g_row0 + ((size_t)a.b * a.H + a.h) * N + a.colbase : nullptr;
      const float gw = (GMODE == 3) ? ((qi == 0) ? a.w_cls2 : a.w_aff2) : a.invH;
      bwd_softmax_tile<GMODE, TAIL>(s, a.tS, a.tDP, a.tDS, a.lane_off, a.half, row, a.colbase, N, grow, cw, gw, a.scale_log2, lse2, dlt, rd_row0,
                                    a.p_row, a.ds_row, pds_par);
    }
    tc::fence_proxy_async_smem();
    tc::mbar_arrive(&s.pds_full);
    if (a.half == 0 && row < 32) BWD_TRACE(1, i, 4);
  }
}

// Work items of the persistent grid: (key tile, head*image).  Full key tiles first, then the thin last tiles (N = p*p+1 leaves
// 17 valid keys in the last tile at 448x448: ~1/3 of the cost), dealt round-robin -- the thin ones starting from the CTAs that
// got one full item less -- so every CTA first runs the <TAIL = false> loops and then the <TAIL = true> ones.
struct Items {
  int kt_full, nfull, nthin;
  __device__ bool at(int c, int G, int k, int& kvt, int& hb, bool& tail) const {
    const int nf = nfull > c ? (nfull - c + G - 1) / G : 0;
    if (k < nf) {
      const int f = c + k * G;
      kvt = f % kt_full;
      hb = f / kt_full;
      tail = false;
      return true;
    }
    k -= nf;
    const int cr = G - 1 - c;
    const int nt = nthin > cr ? (nthin - cr + G - 1) / G : 0;
    if (k < nt) {
      kvt = kt_full;
      hb = cr + k * G;
      tail = true;
      return true;
    }
    return false;
  }
};

// Persistent: one CTA per SM walks over its work items.  The Q/dO ring, the TMEM allocation and every barrier phase run on
// across items, so an item's prologue (TMEM allocation, barrier init, first TMA round trips: 2400 cycles) and epilogue (last dQ
// reduce, dK/dV write-out: 5000 cycles of a 30000-cycle CTA in the one-item-per-CTA version) are paid once per CTA or hidden
// under the next item's first tiles.
__global__ void __launch_bounds__(BWD_THREADS, 1)
attn_bwd_kernel(const __grid_constant__ CUtensorMap tmap_qkv, const __grid_constant__ CUtensorMap tmap_do,
                const __grid_constant__ CUtensorMap tmap_dq,
                const float* __restrict__ lse, const float* __restrict__ delta, const float* __restrict__ g_mean, long long g_bs,
                long long g_ld, GCode gc, __nv_bfloat16* __restrict__ d_qkv, float* __restrict__ g_row0, int* __restrict__ dq_bad, float dq_lim,
                int N, int H, int HB, float scale, float scale_log2) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  BwdSmem& s = *reinterpret_cast<BwdSmem*>(smem_raw);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ntiles = (N + BM - 1) / BM;
  const bool has_code = gc.ptr != nullptr;
  const int G = gridDim.x, cta = blockIdx.x;
  Items items;
  items.kt_full = N / BN;
  items.nfull = items.kt_full * HB;
  items.nthin = (N % BN) ? HB : 0;

  if (warp == 0 && lane == 0) {
    if (tc::smem_u32(smem_raw) & 1023u) __trap();      // SWIZZLE_128B tiles need 1024-byte aligned shared memory
    tc::prefetch_tmap(&tmap_qkv);
    tc::prefetch_tmap(&tmap_do);
    tc::prefetch_tmap(&tmap_dq);
    tc::mbar_init(&s.kv_full, 1);
    tc::mbar_init(&s.kv_empty, 1);
    tc::mbar_init(&s.dkv_free, 128);
    for (int i = 0; i < NST; ++i) {
      tc::mbar_init(&s.qdo_full[i], 1);
      tc::mbar_init(&s.qdo_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) tc::mbar_init(&s.stat_full[i], 64);
    tc::mbar_init(&s.sdp_full, 1);
    tc::mbar_init(&s.sdp_free, 256);
    tc::mbar_init(&s.pds_full, 256);
    tc::mbar_init(&s.pds_free, 1);
    tc::mbar_init(&s.dq_full, 1);
    tc::mbar_init(&s.dq_free, 128);
    tc::fence_barrier_init();
  }
  if (warp == 2) tc::tmem_alloc<512>(&s.tmem_base);
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  if (warp == 0) BWD_TRACE(3, 0, 0);
  const uint32_t tmem = s.tmem_base;
  const uint32_t tS = tmem, tDP = tmem + 128, tDV = tmem + 256, tDK = tmem + 320, tDQ = tmem + 384, tDS = tmem + 448;   // tDS: dS as bf16 (A operand of the dQ MMA)

  if (warp < 4) {
    tc::reg_dealloc<REG_CTRL>();
    if (warp == 0) {
      int T = 0, kvt, hb;
      bool tail;
      for (int k = 0; items.at(cta, G, k, kvt, hb, tail); ++k) {
        const int h = hb % H, b = hb / H, kv0 = kvt * BN;
        tc::mbar_wait(&s.kv_empty, (k & 1) ^ 1);        // every MMA of the previous item has read K / V
        if (tc::elect_one()) {
          tc::mbar_arrive_expect_tx(&s.kv_full, 2 * TILE_BYTES);
          tc::tma_load_4d(s.k, &tmap_qkv, &s.kv_full, 0, H + h, kv0, b);
          tc::tma_load_4d(s.v, &tmap_qkv, &s.kv_full, 0, 2 * H + h, kv0, b);
        }
        __syncwarp();
        for (int i = 0; i < ntiles; ++i, ++T) {
          const int st = T % NST;
          tc::mbar_wait(&s.qdo_empty[st], ((T / NST) & 1) ^ 1);
          if (tc::elect_one()) {
            tc::mbar_arrive_expect_tx(&s.qdo_full[st], 2 * TILE_BYTES);
            tc::tma_load_4d(s.q[st], &tmap_qkv, &s.qdo_full[st], 0, h, i * BM, b);
            tc::tma_load_4d(s.d_o[st], &tmap_do, &s.qdo_full[st], 0, h, i * BM, b);
          }
          __syncwarp();
        }
      }
    } else if (warp == 1) {
      // all 32 lanes walk the loop and wait on the barriers; one elected lane issues (see tc::elect_one)
      // Shared-memory descriptors are built once; a step along K (or to the next 64-wide block) is an addition to the
      // 16-byte-unit start-address field (no carry out of it: every tile lies below 256 KB).
      const uint64_t kd_k = tc::smem_desc_sw128(tc::smem_u32(s.k), 16, 1024);        // K, K-major   (B of S)
      const uint64_t vd_k = tc::smem_desc_sw128(tc::smem_u32(s.v), 16, 1024);        // V, K-major   (B of dP)
      const uint64_t kd_mn = tc::smem_desc_sw128(tc::smem_u32(s.k), 1024, 1024);     // K, MN-major  (B of dQ)
      const uint64_t pd_mn = tc::smem_desc_sw128(tc::smem_u32(s.p[0]), TILE_BYTES, 1024);    // P^T  (A of dV): two 64-wide M blocks 16 KB apart
      const uint64_t dsd_mn = tc::smem_desc_sw128(tc::smem_u32(s.ds[0]), TILE_BYTES, 1024);  // dS^T (A of dK)
      auto issue_scores = [&](int T) {      // S = Q K^T, dP = dO V^T of the CTA's T-th tile
        const int st = T % NST;
        tc::mbar_wait(&s.qdo_full[st], (T / NST) & 1);
        tc::tc_fence_after();
        BWD_TRACE(0, T, 0);
        const uint64_t qd = tc::smem_desc_sw128(tc::smem_u32(s.q[st]), 16, 1024), dod = tc::smem_desc_sw128(tc::smem_u32(s.d_o[st]), 16, 1024);
        if (tc::elect_one()) {
#pragma unroll
          for (int ks = 0; ks < HD / 16; ++ks) tc::mma_ss_off(tS, qd, ks * 2, kd_k, ks * 2, IDESC_S, ks > 0);          // 32 bytes per K step
#pragma unroll
          for (int ks = 0; ks < HD / 16; ++ks) tc::mma_ss_off(tDP, dod, ks * 2, vd_k, ks * 2, IDESC_S, ks > 0);
          tc::tc_commit(&s.sdp_full);
        }
        __syncwarp();
      };
      int T = 0, kvt, hb;
      bool tail;
      for (int k = 0; items.at(cta, G, k, kvt, hb, tail); ++k) {
        tc::mbar_wait(&s.kv_full, k & 1);
        if (T > 0) tc::mbar_wait(&s.sdp_free, (T - 1) & 1);      // the previous item's last tile has left tS / tDP
        issue_scores(T);
        for (int i = 0; i < ntiles; ++i, ++T) {
          const int st = T % NST;
          if (i + 1 < ntiles) {                // scores of the next tile as soon as the softmax warps hold S/dP of this one in registers
            tc::mbar_wait(&s.sdp_free, T & 1);
            issue_scores(T + 1);
          }
          const uint64_t qd_mn = tc::smem_desc_sw128(tc::smem_u32(s.q[st]), 1024, 1024), dod_mn = tc::smem_desc_sw128(tc::smem_u32(s.d_o[st]), 1024, 1024);
          BWD_TRACE(0, T, 1);
          tc::mbar_wait(&s.pds_full, T & 1);                          // P / dS published
          BWD_TRACE(0, T, 2);
          if (T >= 1) tc::mbar_wait(&s.dq_free, (T - 1) & 1);         // the previous dQ has left tDQ
          if (i == 0 && k > 0) tc::mbar_wait(&s.dkv_free, (k - 1) & 1);   // dK / dV of the previous item have left TMEM
          tc::tc_fence_after();
          const uint32_t acc = (i > 0) ? 1u : 0u;
          if (tc::elect_one()) {
#pragma unroll
            for (int ks = 0; ks < BM / 16; ++ks)      // dK += dS^T Q   (M = kv, K = q: 16 q rows = 2048 bytes per step)
              tc::mma_ss_off(tDK, dsd_mn, ks * 128, qd_mn, ks * 128, IDESC_DQ, acc | (ks > 0));
#pragma unroll
            for (int ks = 0; ks < BM / 16; ++ks)      // dV += P^T dO
              tc::mma_ss_off(tDV, pd_mn, ks * 128, dod_mn, ks * 128, IDESC_DQ, acc | (ks > 0));
            tc::tc_commit(&s.pds_free);               // the shared-memory P / dS tiles and Q / dO are free again ...
            tc::tc_commit(&s.qdo_empty[st]);
#pragma unroll
            for (int ks = 0; ks < BN / 16; ++ks)      // dQ_i = dS K   (A = dS out of TMEM: 16 keys = 8 columns per step; B = K MN-major)
              tc::mma_ts_off(tDQ, tDS + ks * 8, kd_mn, ks * 128, IDESC_PV, ks > 0);
            tc::tc_commit(&s.dq_full);                // ... and with dq_full so is tDS
            if (i + 1 == ntiles) tc::tc_commit(&s.kv_empty);   // K / V may be replaced by the next item's
          }
          __syncwarp();
          BWD_TRACE(0, T, 3);
        }
      }
    } else {
      // warps 2, 3: row statistics of the CTA's T-th tile -> s.stat[T & 1] (warp 2: log2-domain LSE, warp 3: delta)
      const int which = warp - 2;
      int T = 0, kvt, hb;
      bool tail;
      for (int k = 0; items.at(cta, G, k, kvt, hb, tail); ++k) {
        const float* src = (which == 0 ? lse : delta) + (size_t)hb * N;       // [B,H,N]: hb = b*H + h
        for (int i = 0; i < ntiles; ++i, ++T) {
          // slot reuse: the gradient MMAs of tile T-2 have retired, so its softmax read the statistics long ago
          if (T >= 2) tc::mbar_wait(&s.qdo_empty[(T - 2) % NST], ((T - 2) / NST) & 1);
          float v[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int qi = i * BM + q * 32 + lane;
            v[q] = (qi < N) ? __ldg(src + qi) : (which == 0 ? INFINITY : 0.f);      // rows past N: P = exp2(-inf) = 0
          }
#pragma unroll
          for (int q = 0; q < 4; ++q) s.stat[T & 1][which][q * 32 + lane] = (which == 0) ? v[q] * kLog2e : v[q];
          tc::mbar_arrive(&s.stat_full[T & 1]);
        }
      }
    }
  } else if (warp < 12) {
    tc::reg_alloc<REG_SOFTMAX>();
    const int we = warp - 4;
    const int row = (warp & 3) * 32 + lane;          // query row inside the tile (TMEM lane)
    const int half = we >> 2;                        // which 64-column (key) half
    const uint32_t lane_off = (uint32_t)((warp & 3) * 32) << 16;
    const float invH = 1.f / (float)H;
    const bool g_vec = (g_mean != nullptr) && ((g_ld & 3) == 0) && ((g_bs & 3) == 0) && ((reinterpret_cast<uintptr_t>(g_mean) & 15) == 0);
    float w_cls2 = 0.f, w_aff2 = 0.f;
    if (has_code) {
      const float sc = gc.scale ? __ldg(gc.scale) : 1.f;
      w_cls2 = 2.f * invH * sc * gc.w_cls;
      w_aff2 = 2.f * invH * sc * gc.w_aff;
    }
    // row start ^ swizzle term (see bwd_softmax_tile)
    const uint32_t swz = (uint32_t)(row & 7) << 4;
    const uint32_t p_row = (tc::smem_u32(s.p[half]) + row * 128) ^ swz, ds_row = (tc::smem_u32(s.ds[half]) + row * 128) ^ swz;
    // one instantiation of the tile loop per (form of G, key-tail) pair; the form of G is fixed per launch and a CTA runs all its
    // full-tile items before its thin ones, so each loop below contains ONE body (with the choice inside the tile loop ptxas
    // hoists the invariants of every body and spills)
    int T = 0, k = 0, kvt, hb;
    bool tail;
    auto run = [&](auto body, bool want_tail) {
      while (items.at(cta, G, k, kvt, hb, tail) && tail == want_tail) {
        const SoftmaxArgs sa{tS, tDP, tDS, lane_off, half, row, kvt * BN + half * 64, N, H, ntiles, hb / H, hb % H, g_mean, g_bs, g_ld, g_row0,
                             gc.ptr, gc.bs, gc.ld, w_cls2, w_aff2, invH, scale_log2, p_row, ds_row, swz};
        body(sa, T);
        T += ntiles;
        ++k;
      }
    };
    if (has_code) {
      run([&](const SoftmaxArgs& sa, int T0) { bwd_softmax_loop<3, false>(s, sa, T0); }, false);
      run([&](const SoftmaxArgs& sa, int T0) { bwd_softmax_loop<3, true>(s, sa, T0); }, true);
    } else if (g_mean != nullptr && g_vec) {
      run([&](const SoftmaxArgs& sa, int T0) { bwd_softmax_loop<2, false>(s, sa, T0); }, false);
      run([&](const SoftmaxArgs& sa, int T0) { bwd_softmax_loop<1, true>(s, sa, T0); }, true);
    } else if (g_mean != nullptr) {
      run([&](const SoftmaxArgs& sa, int T0) { bwd_softmax_loop<1, true>(s, sa, T0); }, false);
      run([&](const SoftmaxArgs& sa, int T0) { bwd_softmax_loop<1, true>(s, sa, T0); }, true);
    } else {
      run([&](const SoftmaxArgs& sa, int T0) { bwd_softmax_loop<0, false>(s, sa, T0); }, false);
      run([&](const SoftmaxArgs& sa, int T0) { bwd_softmax_loop<0, true>(s, sa, T0); }, true);
    }
  } else {
    // drain warpgroup.  Per tile: dQ (rows = queries, 64 d columns) -> 64-bit fixed-point accumulator [B*H, N, 64] (kDqFix) by
    // four TMA reduce-adds of [128 x 16] u64 SWIZZLE_128B boxes, staged alternately in the two 16 KB halves of the staging buffer
    // so that one box is staged while the other is read (rows past N are clipped by the tensor map).  Per item: dV, dK rows
    // (lanes = keys) of the key tile -> d_qkv as bf16 once its last MMA has retired (the last dq_full of the item covers every
    // earlier MMA).
    tc::reg_dealloc<REG_DRAIN>();
    const int row = (warp & 3) * 32 + lane;
    const uint32_t lane_off = (uint32_t)((warp & 3) * 32) << 16;
    const bool leader = (warp == 12 && lane == 0);
    const uint32_t dq_row = (tc::smem_u32(s.dq[0]) + row * 128) ^ ((uint32_t)(row & 7) << 4);      // row start ^ swizzle term
    uint32_t r[32];
    // one box: columns col .. col+15 of query tile i from r[base .. base+15] (fp32) through staging half `buf`.  The box staged
    // there before is the older of the (at most) two in flight: wait until the TMA has read it.
    auto drain_box = [&](int base, int buf, int col, int i, int hb) {
      if (leader) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
      asm volatile("bar.sync 3, 128;" ::: "memory");
      bool bad = false;
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float fa = __uint_as_float(r[base + 2 * e]) * kDqFix, fb = __uint_as_float(r[base + 2 * e + 1]) * kDqFix;
        const bool oka = fabsf(fa) < dq_lim, okb = fabsf(fb) < dq_lim;          // false for NaN too
        bad |= !(oka && okb);
        const long long a = oka ? __float2ll_rn(fa) : 0ll, b = okb ? __float2ll_rn(fb) : 0ll;
        sts128((dq_row + buf * TILE_BYTES) ^ (uint32_t)(e << 4), (uint32_t)a, (uint32_t)((unsigned long long)a >> 32), (uint32_t)b,
               (uint32_t)((unsigned long long)b >> 32));
      }
      if (bad && i * BM + row < N) dq_bad[(size_t)hb * N + i * BM + row] = 1;        // the whole row of dQ comes out as NaN
      tc::fence_proxy_async_smem();
      asm volatile("bar.sync 3, 128;" ::: "memory");
      if (leader) {
        asm volatile("cp.reduce.async.bulk.tensor.3d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(
                         reinterpret_cast<uint64_t>(&tmap_dq)),
                     "r"(tc::smem_u32(s.dq[buf])), "r"(col), "r"(i * BM), "r"(hb)
                     : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      }
    };
    int T = 0, kvt, hb;
    bool tail;
    for (int k = 0; items.at(cta, G, k, kvt, hb, tail); ++k) {
      for (int i = 0; i < ntiles; ++i, ++T) {
        if (warp == 12) BWD_TRACE(2, T, 0);
        tc::mbar_wait(&s.dq_full, T & 1);
        tc::tc_fence_after();
        if (warp == 12) BWD_TRACE(2, T, 1);
        tc::tmem_ld32(tDQ + lane_off, r);
        tc::tmem_ld_wait();
        drain_box(0, 0, 0, i, hb);
        drain_box(16, 1, 16, i, hb);
        tc::tmem_ld32(tDQ + lane_off + 32, r);
        tc::tmem_ld_wait();
        tc::tc_fence_before();
        tc::mbar_arrive(&s.dq_free);                   // tDQ has been read
        if (warp == 12) BWD_TRACE(2, T, 2);
        drain_box(0, 0, 32, i, hb);
        drain_box(16, 1, 48, i, hb);
        if (leader) BWD_TRACE(2, T, 3);
      }
      // dV / dK of this item
      const int h = hb % H, b = hb / H, kv0 = kvt * BN;
      const bool kv_ok = (kv0 + row) < N;
      const size_t E = (size_t)H * HD;
      __nv_bfloat16* base = d_qkv + ((size_t)b * N + min(kv0 + row, N - 1)) * 3 * E + (size_t)h * HD;
#pragma unroll
      for (int part = 0; part < 4; ++part) {           // dV cols 0-31, 32-63, dK cols 0-31, 32-63
        const bool is_k = part >= 2;
        tc::tmem_ld32((is_k ? tDK : tDV) + lane_off + (part & 1) * 32, r);      // warp-collective: outside the per-row validity branch
        tc::tmem_ld_wait();
        if (kv_ok) {
          const float sc = is_k ? scale : 1.f;
          __nv_bfloat16* dst = base + (is_k ? 1 : 2) * E + (part & 1) * 32;
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            uint4 v;
            v.x = tc::pack_bf16(__uint_as_float(r[c * 8 + 0]) * sc, __uint_as_float(r[c * 8 + 1]) * sc);
            v.y = tc::pack_bf16(__uint_as_float(r[c * 8 + 2]) * sc, __uint_as_float(r[c * 8 + 3]) * sc);
            v.z = tc::pack_bf16(__uint_as_float(r[c * 8 + 4]) * sc, __uint_as_float(r[c * 8 + 5]) * sc);
            v.w = tc::pack_bf16(__uint_as_float(r[c * 8 + 6]) * sc, __uint_as_float(r[c * 8 + 7]) * sc);
            reinterpret_cast<uint4*>(dst)[c] = v;
          }
        }
      }
      tc::tc_fence_before();
      tc::mbar_arrive(&s.dkv_free);
    }
    // the TMA reduce-adds are asynchronous: they must complete before the CTA (and its shared memory) goes away
    if (leader) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 0) BWD_TRACE(3, 0, 1);
  if (warp == 2) {
    tc::tc_fence_after();
    tc::tmem_dealloc<512>(tmem);
  }
}

}  // namespace

namespace acr_attn {

int launch_attn_bwd(const CUtensorMap& tmap_qkv, const CUtensorMap& tmap_do, const CUtensorMap& tmap_dq, const float* lse, const float* delta,
                    const float* g_mean, long long g_bs, long long g_ld, const GCode& gc, __nv_bfloat16* d_qkv, float* g_row0,
                    int* dq_bad, int B, int N, int H, float scale, cudaStream_t st) {
  const size_t smem = sizeof(BwdSmem);
  static bool attr_set[64] = {false};
  if (int e = set_max_smem(attn_bwd_kernel, smem, attr_set)) return e;
  static int sms[64] = {0};
  int dev = 0;
  ACR_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64) dev = 0;
  if (!sms[dev]) ACR_CUDA(cudaDeviceGetAttribute(&sms[dev], cudaDevAttrMultiProcessorCount, dev));
  const int kt = (N + BN - 1) / BN;
  const long long nitems = (long long)kt * H * B;
  const unsigned grid = (unsigned)(nitems < sms[dev] ? nitems : sms[dev]);      // persistent: one CTA per SM
  acr::KernelTimer kt_("attn_bwd_kernel", st);
  attn_bwd_kernel<<<grid, BWD_THREADS, smem, st>>>(tmap_qkv, tmap_do, tmap_dq, lse, delta, g_mean, g_bs, g_ld, gc, d_qkv, g_row0, dq_bad,
                                                    dq_fix_limit(kt), N, H, H * B, scale, scale * kLog2e);
  return acr::check_launch("attn_bwd_kernel");
}

}  // namespace acr_attn

#ifdef ACR_BWD_TRACE
extern "C" void acr_bwd_trace_read(unsigned long long* host /* [4*16*8] */) { cudaMemcpyFromSymbol(host, g_bwd_trace, sizeof(g_bwd_trace)); }
#endif
