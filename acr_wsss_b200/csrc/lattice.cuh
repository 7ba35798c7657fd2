// Permutohedral lattice on the GPU, shared by the bilateral filter (bilateral.cu, D = 5) and the dense CRF (densecrf.cu,
// D = 2 and 5).  Device bodies only: each filter owns its kernels, its splat and its slice epilogue, and calls these.
//
// Template parameters:
//   D    feature dimension.  A key is D int16 coordinates packed two per uint32 (D = 5: 3 words, D = 2: 1 word).
//   Pad  which reference `init` the embedding follows:
//          true  the 4-wide SSE init of permutohedral.cpp (bilateral filter): pixels are embedded four at a time and the
//                last group is padded with all-zero feature vectors whose vertices take part in the blur; rounding to
//                the remainder-0 point is nearest-even (_mm_round_ps);
//          false the scalar init of densecrf 2.x (dense CRF): every pixel alone, no pads; rounding compares the two
//                candidate multiples of d+1 and a tie goes to the lower one (`up - e < e - down ? up : down`).
// Everything else (elevation, rank, barycentric weights, keys, blur neighbours, slice) is the same for both.
//
// Data layout in HBM (per image, carved from the caller's workspace; nc = (D+1)*HWp candidates, HWp = HW rounded up to 4
// with pads, HW without):
//   key[NW][nc] u32        packed int16 key of every candidate (k0|k1<<16, k2|k3<<16, k4)
//   bary  [nc] f32         barycentric weight of the candidate
//   table [cap]  i32       open-addressing hash: representative candidate index or -1 (cap = pow2 >= 1.25*nc)
//   rep   [nc] i32         candidate -> representative candidate; `offs` = vertex id + 1 is a separate array
//   vid   [nc] i32         representative candidate -> dense vertex id
//   vcand [nc] i32         vertex id -> representative candidate
//   nbr   [D+1][nc] int2   blur neighbours (vertex id + 1; 0 = missing)
//   val0/val1 [(nc+1) * Kp] f32   lattice values, vertex-major with the Kp = roundup(K, 4) planes contiguous; slot 0 = zeros
// Candidate c = r * HWp + pixel (plane-major: every store of the embedding is coalesced).
#pragma once
#include "common.cuh"
#include <cmath>
#include <type_traits>

namespace acr {
namespace lattice {

template <int D> struct Key { uint32_t w[(D + 1) / 2]; };
template <int D> struct Scales { float s[D]; };

template <typename T>
__device__ __forceinline__ T* img_ptr(T* base, size_t stride_bytes, int n) {
  return reinterpret_cast<T*>(reinterpret_cast<char*>(const_cast<typename std::remove_const<T>::type*>(base)) + stride_bytes * n);
}

// per-image arrays (pointers of image 0; image n lives `ws` bytes further)
template <int D> struct Lattice {
  static constexpr int NW = (D + 1) / 2;
  uint32_t* key[NW];
  float* bary;
  int *table, *rep, *offs, *vid, *vcand, *counter;
  int2* nbr;
  float *val0, *val1;
  uint32_t cap;
  size_t ws;
  int nc, hwp, Kp;
};

template <int D>
__device__ __forceinline__ Lattice<D> for_image(const Lattice<D>& l, int n) {
  Lattice<D> r = l;
#pragma unroll
  for (int i = 0; i < Lattice<D>::NW; ++i) r.key[i] = img_ptr(l.key[i], l.ws, n);
  r.bary = img_ptr(l.bary, l.ws, n);
  r.table = img_ptr(l.table, l.ws, n); r.rep = img_ptr(l.rep, l.ws, n); r.offs = img_ptr(l.offs, l.ws, n);
  r.vid = img_ptr(l.vid, l.ws, n); r.vcand = img_ptr(l.vcand, l.ws, n); r.counter = img_ptr(l.counter, l.ws, n);
  r.nbr = img_ptr(l.nbr, l.ws, n);
  r.val0 = img_ptr(l.val0, l.ws, n); r.val1 = img_ptr(l.val1, l.ws, n);
  return r;
}

template <int D>
__device__ __forceinline__ Key<D> pack_key(const short* k) {
  Key<D> r;
#pragma unroll
  for (int i = 0; i < (D + 1) / 2; ++i)
    r.w[i] = (uint32_t)(uint16_t)k[2 * i] | (2 * i + 1 < D ? ((uint32_t)(uint16_t)k[2 * i + 1] << 16) : 0u);
  return r;
}
template <int D>
__device__ __forceinline__ void unpack_key(const Key<D>& r, short* k) {
#pragma unroll
  for (int i = 0; i < D; ++i) k[i] = (short)((i & 1) ? (r.w[i >> 1] >> 16) : (r.w[i >> 1] & 0xffff));
}
template <int D>
__device__ __forceinline__ bool key_eq(const Key<D>& x, const Key<D>& y) {
  bool e = true;
#pragma unroll
  for (int i = 0; i < (D + 1) / 2; ++i) e = e && x.w[i] == y.w[i];
  return e;
}
// 32-bit mix of the packed key (the reference's multiplicative hash, permutohedral.cpp:42-49, costs five 64-bit multiplies per
// probe; the hash function is free to choose -- results are indexed by key)
template <int D>
__device__ __forceinline__ uint32_t key_hash(const Key<D>& key) {
  uint32_t h = key.w[0] * 0x9E3779B1u;
  if ((D + 1) / 2 > 1) h = (h ^ (h >> 15)) + key.w[1 % ((D + 1) / 2)] * 0x85EBCA77u;
  if ((D + 1) / 2 > 2) h = (h ^ (h >> 13)) + key.w[2 % ((D + 1) / 2)] * 0xC2B2AE3Du;
  h ^= h >> 16;
  return h * 0x27D4EB2Fu;
}
template <int D>
__device__ __forceinline__ Key<D> load_key(const Lattice<D>& l, int c) {
  Key<D> k;
#pragma unroll
  for (int i = 0; i < (D + 1) / 2; ++i) k.w[i] = l.key[i][c];
  return k;
}

// Host: elevation scale factors, permutohedral.cpp:168-171 (densecrf 2.x has the same).
template <int D> Scales<D> scales() {
  Scales<D> sc;
  const float inv_std_dev = (float)(std::sqrt(2.0 / 3.0) * (D + 1));
  for (int i = 0; i < D; ++i) sc.s[i] = (float)(1.0 / std::sqrt((double)((i + 2) * (i + 1))) * inv_std_dev);
  return sc;
}
// Host: slice factor alpha = 1/(1+2^-D), permutohedral.cpp:568.
template <int D> float slice_alpha() { return 1.0f / (1.0f + powf(2.f, -(float)D)); }

// Step 1: per pixel `idx` (< hwp), features f (x/sxy, y/sxy[, r/srgb, g/srgb, b/srgb]) -> D+1 candidate keys + barycentric
// weights.  The same launch clears the hash table and the vertex counter of this image (grid-stride over the table).
// image: this image's [3,H,W] planes (D = 5 only).
template <int D, bool Pad>
__device__ __forceinline__ void embed(const Lattice<D>& lat, const float* __restrict__ image, int H, int W, float sigmargb,
                                      float sigmaxy, const Scales<D>& sc, int idx, int gthreads) {
  constexpr int D1 = D + 1;
  const int HW = H * W;
  for (uint32_t e = idx; e < lat.cap; e += gthreads) lat.table[e] = -1;
  if (idx == 0) *lat.counter = 0;
  if (idx >= lat.hwp) return;
  const int px = idx % W, py = idx / W;
  float f[D];
  if (!Pad || idx < HW) {
    f[0] = __fdiv_rn((float)px, sigmaxy);
    f[1] = __fdiv_rn((float)py, sigmaxy);
#pragma unroll
    for (int i = 2; i < D; ++i) f[i] = __fdiv_rn(__ldg(image + (size_t)(i - 2) * HW + idx), sigmargb);
  } else {
    // The SSE reference embeds pixels four at a time and pads the last group with all-zero feature vectors
    // (permutohedral.cpp:182-186); those phantom pixels still create lattice vertices (:404-413), which
    // take part in the blur.  Reproduce them: keys are inserted, nothing is splatted or sliced.
#pragma unroll
    for (int i = 0; i < D; ++i) f[i] = 0.f;
  }

  float elevated[D1];
  float sm = 0.f;
#pragma unroll
  for (int j = D; j > 0; --j) {
    const float cf = __fmul_rn(f[j - 1], sc.s[j - 1]);
    elevated[j] = __fsub_rn(sm, __fmul_rn((float)j, cf));
    sm = __fadd_rn(sm, cf);
  }
  elevated[0] = sm;

  const float invdplus1 = 1.0f / (float)D1;
  const float dplus1 = (float)D1;
  float rem0[D1], rank[D1];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < D1; ++i) {
    const float v = __fmul_rn(invdplus1, elevated[i]);
    float r;
    if (Pad) {
      r = rintf(v);
    } else {
      const float up = ceilf(v), down = floorf(v);
      r = __fsub_rn(__fmul_rn(up, dplus1), elevated[i]) < __fsub_rn(elevated[i], __fmul_rn(down, dplus1)) ? up : down;
    }
    rem0[i] = __fmul_rn(r, dplus1);
    sum = __fadd_rn(sum, r);
    rank[i] = 0.f;
  }
#pragma unroll
  for (int i = 0; i < D; ++i) {
    const float di = __fsub_rn(elevated[i], rem0[i]);
#pragma unroll
    for (int j = i + 1; j < D1; ++j) {
      const float dj = __fsub_rn(elevated[j], rem0[j]);
      const float c = (di < dj) ? 1.f : 0.f;
      rank[i] += c;
      rank[j] += 1.f - c;
    }
  }
#pragma unroll
  for (int i = 0; i < D1; ++i) {
    rank[i] += sum;
    const float add = (rank[i] < 0.f) ? dplus1 : 0.f;
    const float sub = (rank[i] >= dplus1) ? dplus1 : 0.f;
    rank[i] += add - sub;
    rem0[i] += add - sub;
  }
  float bary[D1 + 1];
#pragma unroll
  for (int i = 0; i < D1 + 1; ++i) bary[i] = 0.f;
#pragma unroll
  for (int i = 0; i < D1; ++i) {
    const float v = __fmul_rn(__fsub_rn(elevated[i], rem0[i]), invdplus1);
    const int p = D - (int)rank[i];
    // dynamic index into a register array: unrolled select keeps it in registers
#pragma unroll
    for (int q = 0; q < D1 + 1; ++q) {
      if (q == p) bary[q] = __fadd_rn(bary[q], v);
      if (q == p + 1) bary[q] = __fsub_rn(bary[q], v);
    }
  }
  bary[0] = __fadd_rn(bary[0], __fadd_rn(1.0f, bary[D1]));

#pragma unroll
  for (int r = 0; r < D1; ++r) {
    short key[D];
#pragma unroll
    for (int i = 0; i < D; ++i) {
      const int rk = (int)rank[i];
      const int canon = (rk <= D - r) ? r : r - D1;     // canonical[r*(d+1) + rk]
      key[i] = (short)((int)rem0[i] + canon);
    }
    const Key<D> k = pack_key<D>(key);
    const size_t c = (size_t)r * lat.hwp + idx;
#pragma unroll
    for (int w = 0; w < Lattice<D>::NW; ++w) lat.key[w][c] = k.w[w];
    lat.bary[c] = bary[r];
  }
}

// Step 2: insert every candidate; the CAS winner of a slot becomes the representative and draws a dense id.
template <int D>
__device__ __forceinline__ int insert_one(const Lattice<D>& lat, const Key<D>& k, uint32_t h, int c) {
  const uint32_t mask = lat.cap - 1;
  h &= mask;
  while (true) {
    int e = ((volatile int*)lat.table)[h];
    if (e == -1) {
      e = atomicCAS(&lat.table[h], -1, c);
      if (e == -1) {
        const int id = atomicAdd(lat.counter, 1);
        lat.vid[c] = id;
        lat.vcand[id] = c;
        return c;
      }
    }
    if (key_eq<D>(load_key(lat, e), k)) return e;
    h = (h + 1) & mask;
  }
}

// Candidate c of a full warp (lanes past nc take part in the warp votes and insert nothing).
template <int D>
__device__ __forceinline__ void insert(const Lattice<D>& lat, int c) {
  const int lane = threadIdx.x & 31;
  const bool valid = c < lat.nc;
  Key<D> k;
#pragma unroll
  for (int i = 0; i < (D + 1) / 2; ++i) k.w[i] = 0u;
  uint32_t h = 0x80000000u | (uint32_t)lane;          // lanes past the end: a group of their own, never inserted
  if (valid) { k = load_key(lat, c); h = key_hash<D>(k) & 0x7fffffffu; }
  // lanes of a warp are consecutive pixels of one remainder plane: most of them share a vertex.  Group by hash, check the key
  // against the group leader's; only leaders (and the rare hash-equal, key-different lane) walk the table.
  const unsigned peers = __match_any_sync(0xffffffffu, h);
  const int leader = __ffs(peers) - 1;
  Key<D> kl;
#pragma unroll
  for (int i = 0; i < (D + 1) / 2; ++i) kl.w[i] = __shfl_sync(0xffffffffu, k.w[i], leader);
  const bool own = valid && (lane == leader || !key_eq<D>(k, kl));
  int res = -1;
  if (own) res = insert_one(lat, k, h, c);
  __syncwarp();
  const int lead_res = __shfl_sync(0xffffffffu, res, leader);
  if (valid) lat.rep[c] = own ? res : lead_res;
}

template <int D>
__device__ __forceinline__ int find(const Lattice<D>& lat, const short* ks) {
  const Key<D> k = pack_key<D>(ks);
  const uint32_t mask = lat.cap - 1;
  uint32_t h = key_hash<D>(k) & 0x7fffffffu & mask;
  while (true) {
    const int e = lat.table[h];
    if (e == -1) return 0;
    if (key_eq<D>(load_key(lat, e), k)) return lat.vid[e] + 1;
    h = (h + 1) & mask;
  }
}

// Step 3 (grid-stride over the image's lattice): blur neighbours of every vertex along each of the d+1 axes and
// candidate -> vertex id + 1.  The caller zero-fills its value arrays in the same launch.
template <int D>
__device__ __forceinline__ void prepare(const Lattice<D>& lat, int t0, int nthreads) {
  constexpr int D1 = D + 1;
  const int M = *lat.counter;
  int* nbr1 = reinterpret_cast<int*>(lat.nbr);
  for (int t = t0; t < M * D1 * 2; t += nthreads) {      // one table lookup per thread step: (vertex, axis, side)
    const int side = t & 1, vj = t >> 1;
    const int v = vj / D1, j = vj - v * D1;
    short key[D], nk[D];
    unpack_key<D>(load_key(lat, lat.vcand[v]), key);
#pragma unroll
    for (int k = 0; k < D; ++k) nk[k] = side ? key[k] + 1 : key[k] - 1;
#pragma unroll
    for (int k = 0; k < D; ++k)
      if (k == j) nk[k] = side ? key[k] - D : key[k] + D;
    nbr1[2 * ((size_t)j * lat.nc + v) + side] = find(lat, nk);
  }
  for (int c = t0; c < lat.nc; c += nthreads) lat.offs[c] = lat.vid[lat.rep[c]] + 1;
}

// Slice of one pixel and 4 planes (quad qq of a Kp-wide value row): alpha * sum_r bary_r * values[vertex_r], in the
// reference's accumulation order.
template <int D>
__device__ __forceinline__ float4 slice_quad(const Lattice<D>& lat, const float* __restrict__ values, int Kp, int pix, int qq,
                                             float alpha) {
  constexpr int D1 = D + 1;
  int o[D1];
  float wt[D1];
#pragma unroll
  for (int r = 0; r < D1; ++r) {
    o[r] = __ldg(lat.offs + (size_t)r * lat.hwp + pix);
    wt[r] = __fmul_rn(__ldg(lat.bary + (size_t)r * lat.hwp + pix), alpha);
  }
  float4 v[D1];
#pragma unroll
  for (int r = 0; r < D1; ++r) v[r] = __ldg(reinterpret_cast<const float4*>(values + (size_t)o[r] * Kp + 4 * qq));
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int r = 0; r < D1; ++r) {
    s.x = __fadd_rn(s.x, __fmul_rn(wt[r], v[r].x));
    s.y = __fadd_rn(s.y, __fmul_rn(wt[r], v[r].y));
    s.z = __fadd_rn(s.z, __fmul_rn(wt[r], v[r].z));
    s.w = __fadd_rn(s.w, __fmul_rn(wt[r], v[r].w));
  }
  return s;
}

// Host: carve one image's lattice from `base` + *off (advanced).  Kp = value row width (planes rounded up to 4).
template <int D, bool Pad>
Lattice<D> carve(void* base, size_t* off, int Kp, int H, int W) {
  Lattice<D> c{};
  const size_t hwp = Pad ? ((size_t)H * W + 3) / 4 * 4 : (size_t)H * W, nc = hwp * (D + 1);
  uint32_t cap = 1;
  while (cap < nc + nc / 4) cap <<= 1;      // worst case (every candidate a distinct vertex): load factor <= 0.8
  c.cap = cap;
  c.nc = (int)nc;
  c.hwp = (int)hwp;
  c.Kp = Kp;
  auto take = [&](size_t bytes) { size_t o = *off; *off += align_up(bytes, 256); return (char*)base + o; };
  c.counter = (int*)take(256);
  for (int i = 0; i < Lattice<D>::NW; ++i) c.key[i] = (uint32_t*)take(nc * sizeof(uint32_t));
  c.bary = (float*)take(nc * sizeof(float));
  c.table = (int*)take((size_t)cap * sizeof(int));
  c.rep = (int*)take(nc * sizeof(int));
  c.offs = (int*)take(nc * sizeof(int));
  c.vid = (int*)take(nc * sizeof(int));
  c.vcand = (int*)take(nc * sizeof(int));
  c.nbr = (int2*)take(nc * (D + 1) * sizeof(int2));
  c.val0 = (float*)take((nc + 1) * Kp * sizeof(float));
  c.val1 = (float*)take((nc + 1) * Kp * sizeof(float));
  return c;
}

}  // namespace lattice
}  // namespace acr
