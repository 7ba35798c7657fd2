// (a1) Fused attention for sm_100a: tcgen05 MMAs with TMEM accumulators, operands staged by TMA (SWIZZLE_128B),
// bf16 in / fp32 accumulate.  Replaces models/vision_transformer.py:203-211 + the head mean of DPT/ACR.py:107-112
// without ever writing the [B,H,N,N] softmax to HBM.
//
// Forward = two kernels per block of the ViT:
//   attn_fwd_kernel  (grid q-tiles x H x B): flash-style S = QK^T -> online softmax -> O = PV, emits O (bf16) and the
//                    per-row log-sum-exp.  P goes registers -> TMEM (bf16) and is the A operand of the PV MMA.
//   attn_mean_kernel (grid kv-tiles x q-tiles x B): loops over the H heads of one 128x128 tile, recomputes S on the
//                    tensor cores, normalises with the LSE, accumulates the head mean in registers and writes the
//                    fp32 tile of A-bar straight into slot l of the [B,L,N,N] stack (coalesced, via smem staging).
//                    Also emits the cls-token row of every head's P (GETAM input).
// N = p*p+1 is never a multiple of 128: TMA zero-fills out-of-range rows, key columns >= N are masked to -inf / 0.
#include "attn_tc.cuh"
#include <cstdlib>

using namespace acr_attn;

namespace {

// ---------------------------------------------------------------------------------------------
struct FwdSmem {
  uint8_t q[TILE_BYTES];
  uint8_t k[2][TILE_BYTES];
  uint8_t v[2][TILE_BYTES];
  float mx[2][2][BM];                // row maxima of the two column halves, double-buffered over key tiles
  float lsum[2][BM];                 // row sums of the two column halves (epilogue)
  uint64_t q_full, kv_full[2], kv_empty[2], s_full, s_free, p_full, o_full;
  uint32_t tmem_base;
};

// 2 CTAs per SM, 384 threads: a control warpgroup (TMA / MMA issue / TMEM alloc) that hands its registers to EIGHT softmax
// warps (setmaxnreg 40 / 96).  A softmax thread owns one query row and 64 of the 128 key columns of a tile (warps 4-7: columns
// 0-63, warps 8-11: columns 64-127; warp % 4 = TMEM lane quadrant), so every scheduler holds four softmax warps (two per
// resident CTA).  Knock-out builds of the previous version (4 softmax warps per CTA, a row x 128 columns per thread: 96 us per
// launch at 16 images) ran in 74 us with BOTH MMAs and all exponentials removed: three quarters of the kernel were the
// ~850-instruction per-tile stream of a warp and its barrier waits with two warps per scheduler to hide them.
//
// Per key tile a thread reads its S columns out of TMEM twice (reads cost ~70 cycles per 64 KB tile): pass 1 for the row
// maximum, exchanged with the partner warp through shared memory, pass 2 for the exponentials; tS is handed back (s_free)
// after the last load of pass 2, so the MMA warp issues S(j+1) under the second half of the exponentials and the P.V MMA.
// (Running the exponentials of tile j ahead of the wait for the P.V MMA of tile j-1, with P(j) held as 32 packed registers and
// only its TMEM stores behind o_full, measured 3 % slower: that chain is not what bounds the tile.)
// O never leaves TMEM during the loop: the P.V MMAs accumulate in place, and a row is rescaled (each warp of a pair takes
// 32 of the 64 columns; warp-uniform decision, identical in both warps) only when its running maximum grew by more than 2^8
// since the last rescale -- P stays <= 2^8, far inside bf16 / fp32 range, and the final O / l is exact whatever stabiliser
// was used.
constexpr float kRescaleThreshold = 8.f;          // log2 units
constexpr int FWD_THREADS = 384;
// named barrier of the two softmax warps that share a lane quadrant (immediate ids: a register id makes ptxas reserve all 16
// barriers of the SM for one CTA)
__device__ __forceinline__ void fwd_pair_sync(int quad) {
  switch (quad) {
    case 0: asm volatile("bar.sync 1, 64;" ::: "memory"); break;
    case 1: asm volatile("bar.sync 2, 64;" ::: "memory"); break;
    case 2: asm volatile("bar.sync 3, 64;" ::: "memory"); break;
    default: asm volatile("bar.sync 4, 64;" ::: "memory"); break;
  }
}
__global__ void __launch_bounds__(FWD_THREADS, 2)
attn_fwd_kernel(const __grid_constant__ CUtensorMap tmap_qkv, __nv_bfloat16* __restrict__ out, float* __restrict__ lse,
                int N, int H, float scale_log2) {
  extern __shared__ uint8_t smem_raw[];
  FwdSmem& s = *reinterpret_cast<FwdSmem*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q0 = blockIdx.x * BM, h = blockIdx.y, b = blockIdx.z;
  const int ntiles = (N + BN - 1) / BN;

  if (warp == 0 && lane == 0) {
    tc::prefetch_tmap(&tmap_qkv);
    tc::mbar_init(&s.q_full, 1);
    for (int i = 0; i < 2; ++i) { tc::mbar_init(&s.kv_full[i], 1); tc::mbar_init(&s.kv_empty[i], 1); }
    tc::mbar_init(&s.s_full, 1);
    tc::mbar_init(&s.s_free, 256);
    tc::mbar_init(&s.p_full, 256);
    tc::mbar_init(&s.o_full, 1);
    tc::fence_barrier_init();
  }
  if (warp == 2) tc::tmem_alloc<256>(&s.tmem_base);
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem = s.tmem_base;
  const uint32_t tS = tmem, tP = tmem + 128, tO = tmem + 192;

  if (warp == 0) {
    tc::reg_dealloc<40>();
    // all lanes wait, one elected lane issues (tc::elect_one: no ELECT/branch loop around every TMA / MMA instruction)
    if (tc::elect_one()) {
      tc::mbar_arrive_expect_tx(&s.q_full, TILE_BYTES);
      tc::tma_load_4d(s.q, &tmap_qkv, &s.q_full, 0, h, q0, b);
    }
    __syncwarp();
    for (int j = 0; j < ntiles; ++j) {
      const int st = j & 1;
      tc::mbar_wait(&s.kv_empty[st], ((j >> 1) & 1) ^ 1);
      if (tc::elect_one()) {
        tc::mbar_arrive_expect_tx(&s.kv_full[st], 2 * TILE_BYTES);
        tc::tma_load_4d(s.k[st], &tmap_qkv, &s.kv_full[st], 0, H + h, j * BN, b);
        tc::tma_load_4d(s.v[st], &tmap_qkv, &s.kv_full[st], 0, 2 * H + h, j * BN, b);
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    tc::reg_dealloc<40>();
    tc::mbar_wait(&s.q_full, 0);
    const uint64_t qd = tc::smem_desc_sw128(tc::smem_u32(s.q), 16, 1024);
    auto issue_s = [&](int j) {
      const uint64_t kd = tc::smem_desc_sw128(tc::smem_u32(s.k[j & 1]), 16, 1024);
      if (tc::elect_one()) {
#pragma unroll
        for (int ks = 0; ks < HD / 16; ++ks) tc::mma_ss_off(tS, qd, ks * 2, kd, ks * 2, IDESC_S, ks > 0);
        tc::tc_commit(&s.s_full);
      }
      __syncwarp();
    };
    tc::mbar_wait(&s.kv_full[0], 0);
    tc::tc_fence_after();
    issue_s(0);
    for (int j = 0; j < ntiles; ++j) {
      const int st = j & 1;
      if (j + 1 < ntiles) {                      // S(j+1) as soon as the softmax warps have read S(j) for the last time
        tc::mbar_wait(&s.kv_full[(j + 1) & 1], ((j + 1) >> 1) & 1);
        tc::mbar_wait(&s.s_free, j & 1);
        tc::tc_fence_after();
        issue_s(j + 1);
      }
      tc::mbar_wait(&s.p_full, j & 1);
      tc::tc_fence_after();
      const uint64_t vd = tc::smem_desc_sw128(tc::smem_u32(s.v[st]), 1024, 1024);
      if (tc::elect_one()) {
#pragma unroll
        for (int ks = 0; ks < BN / 16; ++ks) tc::mma_ts_off(tO, tP + ks * 8, vd, ks * 128, IDESC_PV, (j > 0) || (ks > 0));
        tc::tc_commit(&s.o_full);
        tc::tc_commit(&s.kv_empty[st]);
      }
      __syncwarp();
    }
  } else if (warp < 4) {
    tc::reg_dealloc<40>();
  } else {
    tc::reg_alloc<96>();
    const int half = (warp - 4) >> 2;              // key columns half*64 .. half*64+63 of every tile
    const int quad = warp & 3;                     // TMEM lane quadrant = warp % 4
    const int row = quad * 32 + lane;
    const uint32_t lane_off = (uint32_t)(quad * 32) << 16;
    const int cb = half * 64;
    float m = -INFINITY, l = 0.f;      // m: the stabiliser in use = row max of the RAW scores at the last rescale; l: this half's row sum
    uint32_t r[32];
    // N = p*p+1 leaves a thin last tile: warps whose 32 query rows all lie past N only keep the barrier protocol going
    // (their TMEM lanes hold garbage that is never stored).  Both warps of a pair share their rows, so they agree.
    const bool rows_live = q0 + quad * 32 < N;
    for (int j = 0; j < ntiles; ++j) {
      tc::mbar_wait(&s.s_full, j & 1);
      tc::tc_fence_after();
      if (!rows_live) {
        tc::tc_fence_before();
        tc::mbar_arrive(&s.s_free);
        tc::mbar_arrive(&s.p_full);
        // S(j+1) can complete while the live warps are still on tile j: without this wait the next arrival of this
        // warp would be counted in phase j of p_full and release the P.V MMA before P(j) is complete
        tc::mbar_wait(&s.p_full, j & 1);
        continue;
      }
      const int ncols = min(BN, N - j * BN);         // valid key columns of this tile
      const bool full = (ncols == BN);
      // ---- pass 1: row maximum of this thread's 64 columns
      float mx = -INFINITY;
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        const int c0 = cb + c * 32;
        if (c0 < ncols) {                              // warp-uniform
          tc::tmem_ld32(tS + lane_off + c0, r);
          tc::tmem_ld_wait();
          if (full) {
#pragma unroll
            for (int i = 0; i < 32; ++i) mx = fmaxf(mx, __uint_as_float(r[i]));
          } else {
#pragma unroll
            for (int i = 0; i < 32; ++i) mx = fmaxf(mx, (c0 + i < ncols) ? __uint_as_float(r[i]) : -INFINITY);
          }
        }
      }
      s.mx[j & 1][half][row] = mx;
      fwd_pair_sync(quad);       // the two warps that share these 32 rows
      mx = fmaxf(mx, s.mx[j & 1][half ^ 1][row]);
      // the previous P.V MMA must have retired before tP is rewritten (and before O may be rescaled)
      if (j > 0) {
        tc::mbar_wait(&s.o_full, (j - 1) & 1);
        tc::tc_fence_after();
      }
      if (j == 0) {
        m = mx;
      } else {
        const bool need = (mx - m) * scale_log2 > kRescaleThreshold;
        if (__any_sync(0xffffffffu, need)) {         // rare after the first tiles; warp-collective TMEM access
          const float alpha = need ? tc::fast_exp2((m - mx) * scale_log2) : 1.f;
          if (need) { m = mx; l *= alpha; }
          tc::tmem_ld32(tO + lane_off + half * 32, r);         // this warp's 32 of the 64 columns of O
          tc::tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 32; ++i) r[i] = __float_as_uint(__uint_as_float(r[i]) * alpha);
          tc::tmem_st16(tO + lane_off + half * 32, r);
          tc::tmem_st16(tO + lane_off + half * 32 + 16, r + 16);
        }
      }
      // ---- pass 2: P = exp2(S * scale - m * scale) as bf16 into TMEM, row sum (fp32x2: one FFMA2 + one FADD2 per pair of keys)
      const float ms = m * scale_log2;
      const uint64_t sc2 = tc::f2_pack(scale_log2, scale_log2), nms2 = tc::f2_pack(-ms, -ms);
      uint64_t rs2 = tc::f2_pack(0.f, 0.f);
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        const int c0 = cb + c * 32;
        const bool any = c0 < ncols;                   // warp-uniform
        if (any) {
          tc::tmem_ld32(tS + lane_off + c0, r);
          tc::tmem_ld_wait();
        }
        if (c == 1) {                                  // last read of S(j): tS may be overwritten by S(j+1)
          tc::tc_fence_before();
          tc::mbar_arrive(&s.s_free);
        }
        uint32_t pk[16];
        if (any) {
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            float x0, x1;
            tc::f2_unpack(tc::f2_fma(tc::f2_pack(__uint_as_float(r[2 * i]), __uint_as_float(r[2 * i + 1])), sc2, nms2), x0, x1);
            float p0 = tc::fast_exp2(x0), p1 = tc::fast_exp2(x1);
            if (!full) {                               // keys past N
              if (c0 + 2 * i >= ncols) p0 = 0.f;
              if (c0 + 2 * i + 1 >= ncols) p1 = 0.f;
            }
            rs2 = tc::f2_add(rs2, tc::f2_pack(p0, p1));
            pk[i] = tc::pack_bf16(p0, p1);
          }
        } else {                                       // keys past N: P = 0 (V rows there are zero-filled, 0 * garbage must stay finite)
#pragma unroll
          for (int i = 0; i < 16; ++i) pk[i] = 0u;
        }
        tc::tmem_st16(tP + lane_off + half * 32 + c * 16, pk);
      }
      tc::tmem_st_wait();
      tc::tc_fence_before();
      tc::mbar_arrive(&s.p_full);
      float rs_lo, rs_hi;
      tc::f2_unpack(rs2, rs_lo, rs_hi);
      l += rs_lo + rs_hi;
    }
    if (rows_live) {
      s.lsum[half][row] = l;
      fwd_pair_sync(quad);
      l += s.lsum[half ^ 1][row];
      tc::mbar_wait(&s.o_full, (ntiles - 1) & 1);
      tc::tc_fence_after();
      tc::tmem_ld32(tO + lane_off + half * 32, r);
      tc::tmem_ld_wait();
      if (q0 + row < N) {
        const float inv = 1.f / l;
        __nv_bfloat16* dst = out + ((size_t)b * N + q0 + row) * ((size_t)H * HD) + (size_t)h * HD + half * 32;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          uint4 v;
          v.x = tc::pack_bf16(__uint_as_float(r[c * 8 + 0]) * inv, __uint_as_float(r[c * 8 + 1]) * inv);
          v.y = tc::pack_bf16(__uint_as_float(r[c * 8 + 2]) * inv, __uint_as_float(r[c * 8 + 3]) * inv);
          v.z = tc::pack_bf16(__uint_as_float(r[c * 8 + 4]) * inv, __uint_as_float(r[c * 8 + 5]) * inv);
          v.w = tc::pack_bf16(__uint_as_float(r[c * 8 + 6]) * inv, __uint_as_float(r[c * 8 + 7]) * inv);
          reinterpret_cast<uint4*>(dst)[c] = v;
        }
        if (half == 0) lse[((size_t)b * H + h) * N + q0 + row] = (m * scale_log2 + log2f(l)) * kLn2;
      }
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc::tc_fence_after();
    tc::tmem_dealloc<256>(tmem);
  }
}

// ---------------------------------------------------------------------------------------------
constexpr int MEAN_STAGES = 3;
constexpr int MEAN_SW_SLICES = 4;              // = MEAN_SW / 4 column slices of a tile (declared further down)
struct MeanSmem {
  uint8_t qk[MEAN_STAGES][2][TILE_BYTES];      // [stage][0=Q,1=K]; reused as the fp32 staging tile at the end
  float lse2[MEAN_MAX_H][BM];
  float part[MEAN_SW_SLICES][MEAN_MAX_H][BM];  // MODE 1: per-head row sums of the four column slices (one global atomic per row, head and CTA)
  uint64_t full[MEAN_STAGES], empty[MEAN_STAGES], t_full[2], t_empty[2];
  uint32_t tmem_base;
};
constexpr int STAGE_LD = 129;                  // fp32 staging row stride (conflict-free)
static_assert(sizeof(float) * BM * STAGE_LD <= sizeof(uint8_t) * MEAN_STAGES * 2 * TILE_BYTES, "staging tile must fit");

// MODE 0: mean[b,q,kv] = (1/H) sum_h P_h ; MODE 1 (backward pre-pass): part[kv tile][b,h,q] = (1/H) sum_kv P_h[q,kv] * G[b,q,kv]
// over the CTA's key tile (`mean` is then the read-only G, `p_row0` the partial planes).
// Softmax side: MEAN_SW warps = 4 TMEM lane quadrants x (MEAN_SW / 4) column slices of MEAN_COLS columns; each thread owns
// one query row and MEAN_COLS key columns of the tile.  16 warps (4 per scheduler) instead of 8: the per-head chain
// wait -> tcgen05.ld -> wait -> 32 exponentials of a warp is latency bound (clock64 timeline: 1500 cycles per head against
// ~600 cycles of SFU work with 2 warps per scheduler), more resident warps hide it.
constexpr int MEAN_SW = 16;
static_assert(MEAN_SW == 4 * MEAN_SW_SLICES, "slices of the softmax warps");
constexpr int MEAN_COLS = BN / (MEAN_SW / 4);      // 32
constexpr int MEAN_THREADS = 128 + MEAN_SW * 32;   // 640

template <int MODE>
__global__ void __launch_bounds__(MEAN_THREADS, 1)
attn_mean_kernel(const __grid_constant__ CUtensorMap tmap_qkv, const float* __restrict__ lse, float* __restrict__ mean,
                 long long mean_bs, long long mean_ld, GCode gc, float* __restrict__ p_row0, int N, int H, float scale_log2) {
  extern __shared__ uint8_t smem_raw[];
  MeanSmem& s = *reinterpret_cast<MeanSmem*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int kv0 = blockIdx.x * BN, q0 = blockIdx.y * BM, b = blockIdx.z;

  if (warp == 0 && lane == 0) {
    tc::prefetch_tmap(&tmap_qkv);
    for (int i = 0; i < MEAN_STAGES; ++i) { tc::mbar_init(&s.full[i], 1); tc::mbar_init(&s.empty[i], 1); }
    for (int i = 0; i < 2; ++i) { tc::mbar_init(&s.t_full[i], 1); tc::mbar_init(&s.t_empty[i], MEAN_SW * 32); }
    tc::fence_barrier_init();
  }
  if (warp == 2) tc::tmem_alloc<256>(&s.tmem_base);
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem = s.tmem_base;

  if (warp == 0) {
    for (int h = 0; h < H; ++h) {
      const int st = h % MEAN_STAGES;
      tc::mbar_wait(&s.empty[st], ((h / MEAN_STAGES) & 1) ^ 1);
      if (tc::elect_one()) {
        tc::mbar_arrive_expect_tx(&s.full[st], 2 * TILE_BYTES);
        tc::tma_load_4d(s.qk[st][0], &tmap_qkv, &s.full[st], 0, h, q0, b);
        tc::tma_load_4d(s.qk[st][1], &tmap_qkv, &s.full[st], 0, H + h, kv0, b);
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    for (int h = 0; h < H; ++h) {
      const int st = h % MEAN_STAGES, ab = h & 1;
      tc::mbar_wait(&s.full[st], (h / MEAN_STAGES) & 1);
      tc::mbar_wait(&s.t_empty[ab], ((h >> 1) & 1) ^ 1);
      tc::tc_fence_after();
      const uint64_t qd = tc::smem_desc_sw128(tc::smem_u32(s.qk[st][0]), 16, 1024), kd = tc::smem_desc_sw128(tc::smem_u32(s.qk[st][1]), 16, 1024);
      if (tc::elect_one()) {
#pragma unroll
        for (int ks = 0; ks < HD / 16; ++ks) tc::mma_ss_off(tmem + ab * 128, qd, ks * 2, kd, ks * 2, IDESC_S, ks > 0);
        tc::tc_commit(&s.empty[st]);
        tc::tc_commit(&s.t_full[ab]);
      }
      __syncwarp();
    }
  } else if (warp >= 4) {
    const int we = warp - 4;                       // 0..MEAN_SW-1
    const int row = (warp & 3) * 32 + lane;        // TMEM lane quadrant = warp % 4
    const int slice = we >> 2;                     // which MEAN_COLS-column slice of the tile
    const int sidx = we * 32 + lane;               // 0..MEAN_SW*32-1
    const uint32_t lane_off = (uint32_t)((warp & 3) * 32) << 16;
    const bool row_ok = (q0 + row) < N;
    const int col0 = kv0 + slice * MEAN_COLS;      // first key column of this thread
    float acc[MEAN_COLS];
    const float invH = 1.f / (float)H;
    if (MODE == 0) {
#pragma unroll
      for (int i = 0; i < MEAN_COLS; ++i) acc[i] = 0.f;
    } else if (gc.ptr == nullptr) {
      // G tile of this thread's row, pre-scaled by 1/H; zero outside the map
      const float* grow = mean + (size_t)b * mean_bs + (size_t)(q0 + row) * mean_ld + col0;
#pragma unroll
      for (int i = 0; i < MEAN_COLS; ++i) acc[i] = (row_ok && col0 + i < N) ? __ldg(grow + i) * invH : 0.f;
    } else {
      // sign codes: MEAN_COLS bytes of this row (rows are padded to a multiple of 128 bytes, so the loads stay in bounds)
      const float w2 = gcode_weight(gc, q0 + row, invH);
      const uint4* crow = reinterpret_cast<const uint4*>(gc.ptr + (size_t)b * gc.bs + (size_t)min(q0 + row, N - 1) * gc.ld + col0);
#pragma unroll
      for (int v = 0; v < MEAN_COLS / 16; ++v) {
        const uint4 t = __ldg(crow + v);
        const uint32_t w[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int i = v * 16 + j * 4 + k;
            acc[i] = (row_ok && col0 + i < N) ? ACR_CODE_F(w[j], k) * w2 : 0.f;
          }
      }
    }
    // log2-domain LSE of this tile's rows for every head, staged once: s.lse2[h][row] (+inf for rows past N -> P = 0).
    // The loads of a batch of heads are issued before the first store (this sits on the CTA's critical path).
    {
      constexpr int HSTEP = MEAN_SW * 32 / BM;     // heads covered per pass of all softmax threads
      const int rr = sidx & (BM - 1);
      const bool ok = (q0 + rr) < N;
      const float* lp = lse + (size_t)b * H * N + q0 + rr;
      for (int h0 = sidx / BM; h0 < H; h0 += HSTEP * 4) {
        float v[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) v[k] = (ok && h0 + HSTEP * k < H) ? __ldg(lp + (size_t)(h0 + HSTEP * k) * N) : INFINITY;
#pragma unroll
        for (int k = 0; k < 4; ++k)
          if (h0 + HSTEP * k < H) s.lse2[h0 + HSTEP * k][rr] = v[k] * kLog2e;
      }
    }
    asm volatile("bar.sync 1, %0;" ::"n"(MEAN_SW * 32) : "memory");
    const bool tail = (kv0 + BN > N);
    const bool row0_warp = (MODE == 0) && (p_row0 != nullptr) && (q0 == 0) && ((warp & 3) == 0);
    // thin last tiles (N = p*p+1): warps whose 32 rows or columns all lie past N only keep the barrier protocol going
    const bool live = (q0 + (warp & 3) * 32 < N) && (col0 < N);
    uint32_t r[32];
    for (int h = 0; h < H; ++h) {
      const int ab = h & 1;
      const float lse2 = s.lse2[h][row];
      tc::mbar_wait(&s.t_full[ab], (h >> 1) & 1);
      tc::tc_fence_after();
      float part = 0.f;
#pragma unroll
      for (int c = 0; c < MEAN_COLS / 32; ++c) {
        const int colbase = col0 + c * 32;
        if (!live || (tail && colbase >= N)) break;
        tc::tmem_ld32(tmem + ab * 128 + lane_off + slice * MEAN_COLS + c * 32, r);
        tc::tmem_ld_wait();
        if (!tail) {               // fp32x2: 16 FFMA2 + 32 MUFU.EX2 + 16 FADD2 (or FFMA2) per head and thread
          const uint64_t sc2 = tc::f2_pack(scale_log2, scale_log2), nl2 = tc::f2_pack(-lse2, -lse2);
          uint64_t part2 = tc::f2_pack(0.f, 0.f);
#pragma unroll
          for (int i = 0; i < 32; i += 2) {
            float x0, x1;
            tc::f2_unpack(tc::f2_fma(tc::f2_pack(__uint_as_float(r[i]), __uint_as_float(r[i + 1])), sc2, nl2), x0, x1);
            const float p0 = tc::fast_exp2(x0), p1 = tc::fast_exp2(x1);
            const uint64_t pp = tc::f2_pack(p0, p1), aa = tc::f2_pack(acc[c * 32 + i], acc[c * 32 + i + 1]);
            if (MODE == 0) {
              tc::f2_unpack(tc::f2_add(aa, pp), acc[c * 32 + i], acc[c * 32 + i + 1]);
              r[i] = __float_as_uint(p0); r[i + 1] = __float_as_uint(p1);
            } else {
              part2 = tc::f2_fma(pp, aa, part2);
            }
          }
          if (MODE == 1) { float a0, a1; tc::f2_unpack(part2, a0, a1); part += a0 + a1; }
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            float p = tc::fast_exp2(fmaf(__uint_as_float(r[i]), scale_log2, -lse2));
            if (colbase + i >= N) p = 0.f;
            if (MODE == 0) { acc[c * 32 + i] += p; r[i] = __float_as_uint(p); } else part = fmaf(p, acc[c * 32 + i], part);
          }
        }
        if (row0_warp && lane == 0) {       // cls-token row of this head's P (GETAM input)
          float* dst0 = p_row0 + ((size_t)b * H + h) * N + colbase;
#pragma unroll
          for (int i = 0; i < 32; ++i)
            if (colbase + i < N) dst0[i] = __uint_as_float(r[i]);
        }
      }
      tc::tc_fence_before();
      tc::mbar_arrive(&s.t_empty[ab]);
      if (MODE == 1) s.part[slice][h][row] = part;
    }
    if (MODE == 1) {
      // this key tile's share of delta[b,h,q] (the four slices' sums) -> partial plane blockIdx.x, one store per (row, head) of the
      // CTA after the head loop; bwd_delta_kernel adds the planes in key-tile order (a float atomic here would make the sum's
      // rounding depend on which CTA lands first)
      asm volatile("bar.sync 1, %0;" ::"n"(MEAN_SW * 32) : "memory");
      float* plane = p_row0 + (size_t)blockIdx.x * gridDim.z * H * N;
      for (int idx = sidx; idx < H * BM; idx += MEAN_SW * 32) {
        const int hh = idx / BM, rr = idx % BM;
        if (q0 + rr < N) {
          float v = 0.f;
#pragma unroll
          for (int sl = 0; sl < MEAN_SW_SLICES; ++sl) v += s.part[sl][hh][rr];
          plane[((size_t)b * H + hh) * N + q0 + rr] = v;
        }
      }
    }
    if (MODE == 0) {
    // All MMAs have completed (the last t_full was observed) and every TMA load was consumed: the pipeline
    // buffers are free -> stage the tile so that global stores are row-contiguous.
    float* stage = reinterpret_cast<float*>(&s.qk[0][0][0]);
#pragma unroll
    for (int i = 0; i < MEAN_COLS; ++i) stage[row * STAGE_LD + slice * MEAN_COLS + i] = acc[i] * invH;
    asm volatile("bar.sync 1, %0;" ::"n"(MEAN_SW * 32) : "memory");
    // each warp writes BM / MEAN_SW rows, 4 at a time: 16 shared loads in flight before the 16 (row-contiguous, 128-byte) stores
    float* dst = mean + (size_t)b * mean_bs;
    constexpr int RPW = BM / MEAN_SW;
#pragma unroll 1
    for (int r4 = we * RPW; r4 < we * RPW + RPW; r4 += 4) {
      if (q0 + r4 >= N) break;
      float v[4][4];
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int cc = 0; cc < 4; ++cc) v[u][cc] = stage[(r4 + u) * STAGE_LD + cc * 32 + lane];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        if (q0 + r4 + u < N) {
#pragma unroll
          for (int cc = 0; cc < 4; ++cc) {
            const int col = cc * 32 + lane;
            if (kv0 + col < N) dst[(size_t)(q0 + r4 + u) * N + kv0 + col] = v[u][cc];
          }
        }
      }
    }
    }  // MODE == 0
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc::tc_fence_after();
    tc::tmem_dealloc<256>(tmem);
  }
}

// ---------------------------------------------------------------------------------------------
}  // namespace

namespace acr_attn {
EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess || qres != cudaDriverEntryPointSuccess)
      return nullptr;
    fn = (EncodeTiledFn)p;
  }
  return fn;
}

int make_tmap(CUtensorMap* m, const void* base, int B, int N, int SH, int D) {
  EncodeTiledFn fn = get_encode_fn();
  ACR_REQUIRE(fn != nullptr, ACR_E_NOSM100, "cuTensorMapEncodeTiled unavailable");
  cuuint64_t dims[4] = {(cuuint64_t)D, (cuuint64_t)SH, (cuuint64_t)N, (cuuint64_t)B};
  cuuint64_t strides[3] = {(cuuint64_t)D * 2, (cuuint64_t)SH * D * 2, (cuuint64_t)N * SH * D * 2};
  cuuint32_t box[4] = {(cuuint32_t)D, 1, (cuuint32_t)BM, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  ACR_REQUIRE(r == CUDA_SUCCESS, ACR_E_INVAL, "cuTensorMapEncodeTiled failed (%d)", (int)r);
  return 0;
}

}  // namespace acr_attn

extern "C" int acr_attn_fwd_bf16(const void* qkv, int B, int N, int H, int D, float scale,
                                 void* out, float* lse, float* attn_mean, long long mean_batch_stride,
                                 float* p_row0, void* stream) {
  ACR_REQUIRE(qkv && out && lse, ACR_E_INVAL, "acr_attn_fwd_bf16: null pointer");
  ACR_REQUIRE(B > 0 && N > 0 && H > 0, ACR_E_INVAL, "acr_attn_fwd_bf16: bad shape");
  ACR_REQUIRE(D == HD, ACR_E_INVAL, "acr_attn_fwd_bf16: head dim %d unsupported (64 only)", D);
  ACR_REQUIRE(B <= 65535 && H <= MEAN_MAX_H, ACR_E_INVAL, "acr_attn_fwd_bf16: B <= 65535 and H <= %d required", MEAN_MAX_H);
  ACR_REQUIRE(((uintptr_t)qkv & 15) == 0 && ((uintptr_t)out & 15) == 0, ACR_E_ALIGN, "acr_attn_fwd_bf16: qkv/out must be 16-byte aligned");
  ACR_REQUIRE(p_row0 == nullptr || attn_mean != nullptr, ACR_E_INVAL, "acr_attn_fwd_bf16: p_row0 needs attn_mean");
  ACR_REQUIRE(acr_device_is_sm100(), ACR_E_NOSM100, "acr_attn_fwd_bf16: needs an sm_100 device");
  cudaStream_t st = (cudaStream_t)stream;
  CUtensorMap tmap;
  if (int e = make_tmap(&tmap, qkv, B, N, 3 * H, D)) return e;
  const float scale_log2 = scale * kLog2e;
  const int qt = (N + BM - 1) / BM, kt = (N + BN - 1) / BN;
  {
    const size_t smem = sizeof(FwdSmem) + 1024;
    static bool attr_set[64] = {false};
    if (int e = set_max_smem(attn_fwd_kernel, smem, attr_set)) return e;
    dim3 grid(qt, H, B);
    acr::KernelTimer kt_("attn_fwd_kernel", st);
    attn_fwd_kernel<<<grid, FWD_THREADS, smem, st>>>(tmap, (__nv_bfloat16*)out, lse, N, H, scale_log2);
    if (int e = acr::check_launch("attn_fwd_kernel")) return e;
  }
  if (attn_mean) {
    const size_t smem = sizeof(MeanSmem) + 1024;
    static bool attr_set[64] = {false};
    if (int e = set_max_smem(attn_mean_kernel<0>, smem, attr_set)) return e;
    dim3 grid(kt, qt, B);
    acr::KernelTimer kt_("attn_mean_kernel", st);
    attn_mean_kernel<0><<<grid, MEAN_THREADS, smem, st>>>(tmap, lse, attn_mean, mean_batch_stride, (long long)N, GCode{}, p_row0, N, H, scale_log2);
    if (int e = acr::check_launch("attn_mean_kernel")) return e;
  }
  return 0;
}


// =============================================================================================
// Backward.  dP_h = dO_h V_h^T + G/H ; dS_h = P_h * (dP_h - delta) ; delta[q] = sum_j P_h[q,j] dP_h[q,j]
//   = dO_q . O_q + (1/H) sum_j P_h[q,j] G[q,j]   (the second term is what the affinity gradient adds).
// Kernels: attn_mean_kernel<1> (P.G/H per key tile) -> bwd_delta_kernel (dO.O + the key tiles' P.G/H in order, zero-fill of
// the dQ accumulator) -> attn_bwd_kernel (attn_bwd_tc.cu: persistent, rows = queries, dQ tiles reduced across kv tiles by TMA
// reduce-adds in 64-bit fixed point) -> bwd_dq_convert_kernel.  Every sum has a fixed order or is exact: same result every run.
// =============================================================================================
namespace {


__global__ void __launch_bounds__(256)
bwd_delta_kernel(const __nv_bfloat16* __restrict__ out, const __nv_bfloat16* __restrict__ d_out, const float* __restrict__ part,
                 int nparts, float* __restrict__ delta, float4* __restrict__ dq_acc, int* __restrict__ dq_bad, long long rows, int N, int H) {
  // delta[b,h,n] = dO[b,n,h,:] . O[b,n,h,:] + part[0][b,h,n] + ... + part[nparts-1][b,h,n].  A warp takes 4 consecutive (b,n,h)
  // rows at a time: 8 lanes x 16 bytes per 128-byte row (fully coalesced 512-byte requests), 3 shuffles.  The same pass zeroes
  // the 64-bit dQ accumulator the backward kernel reduces into (64 values per row) and its row flags, which saves a separate
  // memset node per block of the ViT.
  const int lane = threadIdx.x & 31;
  const long long t = ((long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * 4 + (lane >> 3);
  const bool ok = t < rows;
  float acc = 0.f;
  if (ok) {
    const uint4 a = __ldg(reinterpret_cast<const uint4*>(out + t * HD) + (lane & 7));
    const uint4 d = __ldg(reinterpret_cast<const uint4*>(d_out + t * HD) + (lane & 7));
    const __nv_bfloat162* a2 = reinterpret_cast<const __nv_bfloat162*>(&a);
    const __nv_bfloat162* d2 = reinterpret_cast<const __nv_bfloat162*>(&d);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float2 fa = __bfloat1622float2(a2[i]), fd = __bfloat1622float2(d2[i]);
      acc = fmaf(fa.x, fd.x, acc);
      acc = fmaf(fa.y, fd.y, acc);
    }
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int m = 0; m < 4; ++m) dq_acc[t * (HD / 2) + m * 8 + (lane & 7)] = z;
  }
  acc += __shfl_xor_sync(0xffffffffu, acc, 1);
  acc += __shfl_xor_sync(0xffffffffu, acc, 2);
  acc += __shfl_xor_sync(0xffffffffu, acc, 4);
  if (ok && (lane & 7) == 0) {
    const int h = (int)(t % H);
    const long long bn = t / H;
    const int n = (int)(bn % N), b = (int)(bn / N);
    const size_t idx = ((size_t)b * H + h) * N + n;
    for (int k = 0; k < nparts; ++k) acc += __ldg(part + (size_t)k * rows + idx);
    delta[idx] = acc;
    dq_bad[idx] = 0;
  }
}

__global__ void __launch_bounds__(256)
bwd_dq_convert_kernel(const long long* __restrict__ dq_acc, const int* __restrict__ dq_bad, __nv_bfloat16* __restrict__ d_qkv, int B, int N,
                      int H, float scale) {
  // dq_acc [B,H,N,64] 64-bit fixed point -> d_qkv[b,n,0,h,:] bf16 (scaled), NaN for a row whose sum left the fixed-point range
  // or met a non-finite value (dq_bad); one thread per 8 elements
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)B * H * N * (HD / 8)) return;
  const int c = (int)(t % (HD / 8));
  const long long row = t / (HD / 8);               // (b*H + h)*N + n
  const int n = (int)(row % N);
  const int h = (int)((row / N) % H);
  const int b = (int)(row / ((long long)N * H));
  const longlong2* src = reinterpret_cast<const longlong2*>(dq_acc + row * HD + c * 8);
  const float sc = __ldg(dq_bad + row) ? __int_as_float(0x7fc00000) : scale * kDqUnfix;    // kDqUnfix * scale is exact
  float x[8];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const longlong2 q = __ldg(src + j);
    x[2 * j] = __ll2float_rn(q.x) * sc;
    x[2 * j + 1] = __ll2float_rn(q.y) * sc;
  }
  uint4 v;
  v.x = tc::pack_bf16(x[0], x[1]);
  v.y = tc::pack_bf16(x[2], x[3]);
  v.z = tc::pack_bf16(x[4], x[5]);
  v.w = tc::pack_bf16(x[6], x[7]);
  *reinterpret_cast<uint4*>(d_qkv + (((size_t)b * N + n) * 3 + 0) * ((size_t)H * HD) + (size_t)h * HD + c * 8) = v;
}

}  // namespace

extern "C" size_t acr_attn_bwd_bf16_workspace(int B, int N, int H, int D) {
  if (B <= 0 || N <= 0 || H <= 0 || D <= 0) return 0;
  const size_t rows = (size_t)B * H * N, kt = (N + BN - 1) / BN;
  // delta | 64-bit dQ accumulator | one delta partial plane per key tile | dQ row flags
  return acr::align_up(rows * sizeof(float), 256) + acr::align_up(rows * D * sizeof(long long), 256) + acr::align_up(kt * rows * sizeof(float), 256) +
         acr::align_up(rows * sizeof(int), 256);
}

extern "C" int acr_attn_bwd_bf16(const void* qkv, const void* out, const float* lse, const void* d_out,
                                 int B, int N, int H, int D, float scale,
                                 const float* g_mean, long long g_batch_stride, long long g_row_stride,
                                 const unsigned char* g_code, long long code_batch_stride, long long code_row_stride,
                                 float w_cls, float w_aff, const float* g_scale,
                                 void* d_qkv, float* g_row0, void* workspace, size_t workspace_bytes, void* stream) {
  ACR_REQUIRE(qkv && out && lse && d_out && d_qkv && workspace, ACR_E_INVAL, "acr_attn_bwd_bf16: null pointer");
  ACR_REQUIRE(B > 0 && N > 0 && H > 0, ACR_E_INVAL, "acr_attn_bwd_bf16: bad shape");
  ACR_REQUIRE(D == HD, ACR_E_INVAL, "acr_attn_bwd_bf16: head dim %d unsupported (64 only)", D);
  ACR_REQUIRE(B <= 65535 && H <= MEAN_MAX_H, ACR_E_INVAL, "acr_attn_bwd_bf16: B <= 65535 and H <= %d required", MEAN_MAX_H);
  ACR_REQUIRE(g_mean == nullptr || g_row_stride >= N, ACR_E_INVAL, "acr_attn_bwd_bf16: g_row_stride < N");
  ACR_REQUIRE(g_mean == nullptr || g_code == nullptr, ACR_E_INVAL, "acr_attn_bwd_bf16: give g_mean OR g_code");
  ACR_REQUIRE(g_code == nullptr || ((code_row_stride % 128) == 0 && code_row_stride >= (long long)((N + 127) / 128) * 128 &&
                                    (code_batch_stride % 16) == 0 && ((uintptr_t)g_code & 15) == 0),
              ACR_E_ALIGN, "acr_attn_bwd_bf16: g_code rows must be 128-byte padded and 16-byte aligned");
  const GCode gc{g_code, code_batch_stride, code_row_stride, w_cls, w_aff, g_scale};
  ACR_REQUIRE(((uintptr_t)qkv & 15) == 0 && ((uintptr_t)out & 15) == 0 && ((uintptr_t)d_out & 15) == 0 && ((uintptr_t)d_qkv & 15) == 0,
              ACR_E_ALIGN, "acr_attn_bwd_bf16: tensors must be 16-byte aligned");
  ACR_REQUIRE(((uintptr_t)workspace & 255) == 0, ACR_E_ALIGN, "acr_attn_bwd_bf16: workspace must be 256-byte aligned");
  ACR_REQUIRE(workspace_bytes >= acr_attn_bwd_bf16_workspace(B, N, H, D), ACR_E_NOMEM, "acr_attn_bwd_bf16: workspace too small");
  ACR_REQUIRE(acr_device_is_sm100(), ACR_E_NOSM100, "acr_attn_bwd_bf16: needs an sm_100 device");
  cudaStream_t st = (cudaStream_t)stream;
  const size_t rows = (size_t)B * H * N;
  const int qt = (N + BM - 1) / BM, kt = (N + BN - 1) / BN;
  float* delta = (float*)workspace;
  long long* dq_acc = (long long*)((char*)workspace + acr::align_up(rows * sizeof(float), 256));
  float* delta_part = (float*)((char*)dq_acc + acr::align_up(rows * D * sizeof(long long), 256));
  int* dq_bad = (int*)((char*)delta_part + acr::align_up((size_t)kt * rows * sizeof(float), 256));
  CUtensorMap tmap_qkv, tmap_do, tmap_dq;
  if (int e = make_tmap(&tmap_qkv, qkv, B, N, 3 * H, D)) return e;
  if (int e = make_tmap(&tmap_do, d_out, B, N, H, D)) return e;
  {   // 64-bit dQ accumulator [B*H, N, 64] as (d, n, bh); box = 16 values (128 B, SWIZZLE_128B) x 128 rows
    EncodeTiledFn fn = get_encode_fn();
    ACR_REQUIRE(fn != nullptr, ACR_E_NOSM100, "cuTensorMapEncodeTiled unavailable");
    cuuint64_t dims[3] = {(cuuint64_t)HD, (cuuint64_t)N, (cuuint64_t)B * H};
    cuuint64_t strides[2] = {(cuuint64_t)HD * 8, (cuuint64_t)N * HD * 8};
    cuuint32_t box[3] = {16, (cuuint32_t)BM, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = fn(&tmap_dq, CU_TENSOR_MAP_DATA_TYPE_UINT64, 3, dq_acc, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    ACR_REQUIRE(r == CUDA_SUCCESS, ACR_E_INVAL, "cuTensorMapEncodeTiled(dq) failed (%d)", (int)r);
  }
  const float scale_log2 = scale * kLog2e;

  const bool with_g = g_mean || g_code;
  if (with_g) {
    const size_t smem = sizeof(MeanSmem) + 1024;
    static bool attr_set[64] = {false};
    if (int e = set_max_smem(attn_mean_kernel<1>, smem, attr_set)) return e;
    dim3 grid(kt, qt, B);
    acr::KernelTimer kt_("attn_delta_kernel", st);
    attn_mean_kernel<1><<<grid, MEAN_THREADS, smem, st>>>(tmap_qkv, lse, const_cast<float*>(g_mean), g_batch_stride, g_row_stride, gc, delta_part, N, H, scale_log2);
    if (int e = acr::check_launch("attn_mean_kernel<1>")) return e;
  }
  bwd_delta_kernel<<<(unsigned)((rows + 31) / 32), 256, 0, st>>>((const __nv_bfloat16*)out, (const __nv_bfloat16*)d_out, delta_part,
                                                               with_g ? kt : 0, delta, reinterpret_cast<float4*>(dq_acc), dq_bad, (long long)rows, N, H);
  if (int e = acr::check_launch("bwd_delta_kernel")) return e;
  if (int e = launch_attn_bwd(tmap_qkv, tmap_do, tmap_dq, lse, delta, g_mean, g_batch_stride, g_row_stride, gc, (__nv_bfloat16*)d_qkv, g_row0, dq_bad, B, N, H, scale, st))
    return e;
  const long long nconv = (long long)rows * (HD / 8);
  bwd_dq_convert_kernel<<<(unsigned)((nconv + 255) / 256), 256, 0, st>>>(dq_acc, dq_bad, (__nv_bfloat16*)d_qkv, B, N, H, scale);
  return acr::check_launch("bwd_dq_convert_kernel");
}
