/*
 * permuto_oracle.c -- CPU ORACLE (test infrastructure only) for the permutohedral bilateral filter.
 *
 * A scalar restatement of the reference's algorithm as the x86-64 build executes it (the SSE branch,
 * wrapper/bilateralfilter/permutohedral.cpp:115-316 init, :507-583 compute; features and the per-image /
 * per-plane loops from bilateralfilter.cpp:4-55).  Written from the algorithm description, NOT copied:
 * one pixel at a time instead of four, own hash map, all K planes share one lattice build.
 * Must be compiled with -ffp-contract=off (the SSE code has separate multiply and add roundings).
 *
 * Parity status: pinned by execution against oracle/_ref (the reference's own C++ compiled from
 * /root/reference by oracle/Makefile) in tests/test_oracle_golden.py, and by tests/golden/bilateral_*.npz.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define DF 5            /* feature dimension d            */
#define DV (DF + 1)     /* vertices per simplex, d + 1    */

typedef struct { int16_t k[DF]; } key_t_;

typedef struct {
  size_t cap, filled;
  int* slots;           /* vertex id or -1 */
  key_t_* keys;         /* by vertex id    */
} map_t;

static uint64_t key_hash(const int16_t* k) {
  uint64_t r = 0;
  for (int i = 0; i < DF; i++) { r += (uint64_t)(int64_t)k[i]; r *= 1664525u; }   /* permutohedral.cpp:42-49 */
  return r;
}

static int map_find(map_t* m, const int16_t* k, int create) {
  size_t h = key_hash(k) % m->cap;
  for (;;) {
    int e = m->slots[h];
    if (e < 0) {
      if (!create) return -1;
      memcpy(m->keys[m->filled].k, k, sizeof(int16_t) * DF);
      m->slots[h] = (int)m->filled;
      return (int)m->filled++;
    }
    if (memcmp(m->keys[e].k, k, sizeof(int16_t) * DF) == 0) return e;
    if (++h == m->cap) h = 0;
  }
}

/* Embed one feature vector: writes DV keys and DV barycentric weights (permutohedral.cpp:188-257). */
static void embed(const float* f, const float* scale, int16_t keys[DV][DF], float bary_out[DV]) {
  float elevated[DV], rem0[DV], rank[DV], bary[DV + 1];
  const float invdp1 = 1.0f / (float)DV, dp1 = (float)DV;
  float sm = 0.f;
  for (int j = DF; j > 0; j--) {
    float cf = f[j - 1] * scale[j - 1];
    elevated[j] = sm - (float)j * cf;
    sm += cf;
  }
  elevated[0] = sm;
  float sum = 0.f;
  for (int i = 0; i < DV; i++) {
    float v = nearbyintf(invdp1 * elevated[i]);     /* round-to-nearest-even, as cvtps / _mm_round_ps */
    rem0[i] = v * dp1;
    sum += v;
    rank[i] = 0.f;
  }
  for (int i = 0; i < DF; i++) {
    float di = elevated[i] - rem0[i];
    for (int j = i + 1; j < DV; j++) {
      float dj = elevated[j] - rem0[j];
      float c = (di < dj) ? 1.f : 0.f;
      rank[i] += c;
      rank[j] += 1.f - c;
    }
  }
  for (int i = 0; i < DV; i++) {
    rank[i] += sum;
    float add = (rank[i] < 0.f) ? dp1 : 0.f;
    float sub = (rank[i] >= dp1) ? dp1 : 0.f;
    rank[i] += add - sub;
    rem0[i] += add - sub;
  }
  for (int i = 0; i < DV + 1; i++) bary[i] = 0.f;
  for (int i = 0; i < DV; i++) {
    float v = (elevated[i] - rem0[i]) * invdp1;
    int p = DF - (int)rank[i];
    bary[p] += v;
    bary[p + 1] -= v;
  }
  bary[0] += 1.0f + bary[DV];
  for (int r = 0; r < DV; r++) {
    for (int i = 0; i < DF; i++) {
      int rk = (int)rank[i];
      int canon = (rk <= DF - r) ? r : r - DV;      /* canonical simplex, permutohedral.cpp:160-165 */
      keys[r][i] = (int16_t)(rem0[i] + (float)canon);
    }
    bary_out[r] = bary[r];
  }
}

/* One image: image [3,H,W] in 0..255, in/out [K,H,W].  Returns the number of lattice vertices M (K = 0: the lattice only,
 * in/out are not read).  skip_blur_axis in 0..DF leaves that one of the d+1 blur passes out -- a deliberately wrong filter
 * the tests use to show that they notice a missing pass; -1 is the filter. */
int permuto_oracle_image_variant(const float* image, const float* in, float* out, int K, int H, int W,
                                 float sigmargb, float sigmaxy, int skip_blur_axis) {
  const int HW = H * W, HWpad = (HW + 3) / 4 * 4;   /* the reference pads the last group of 4 with zero features */
  float scale[DF];
  const float inv_std_dev = (float)(sqrt(2.0 / 3.0) * (DF + 1));
  for (int i = 0; i < DF; i++) scale[i] = (float)(1.0 / sqrt((double)((i + 2) * (i + 1))) * inv_std_dev);

  map_t m;
  m.cap = (size_t)HWpad * DV * 2 + 16;
  m.filled = 0;
  m.slots = (int*)malloc(m.cap * sizeof(int));
  m.keys = (key_t_*)malloc((size_t)HWpad * DV * sizeof(key_t_));
  memset(m.slots, 0xff, m.cap * sizeof(int));
  int* offs = (int*)malloc((size_t)HWpad * DV * sizeof(int));
  float* bary = (float*)malloc((size_t)HWpad * DV * sizeof(float));

  for (int idx = 0; idx < HWpad; idx++) {
    float f[DF] = {0.f, 0.f, 0.f, 0.f, 0.f};
    if (idx < HW) {
      int x = idx % W, y = idx / W;
      f[0] = (float)x / sigmaxy;                    /* bilateralfilter.cpp:8-16 */
      f[1] = (float)y / sigmaxy;
      f[2] = image[idx] / sigmargb;
      f[3] = image[HW + idx] / sigmargb;
      f[4] = image[2 * HW + idx] / sigmargb;
    }
    int16_t keys[DV][DF];
    float b[DV];
    embed(f, scale, keys, b);
    for (int r = 0; r < DV; r++) {
      offs[(size_t)idx * DV + r] = map_find(&m, keys[r], 1);
      bary[(size_t)idx * DV + r] = b[r];
    }
  }
  const int M = (int)m.filled;

  int* n1 = (int*)malloc((size_t)M * DV * sizeof(int));
  int* n2 = (int*)malloc((size_t)M * DV * sizeof(int));
  for (int j = 0; j < DV; j++) {
    for (int v = 0; v < M; v++) {
      int16_t a[DF], b[DF];
      for (int k = 0; k < DF; k++) { a[k] = m.keys[v].k[k] - 1; b[k] = m.keys[v].k[k] + 1; }
      if (j < DF) { a[j] = m.keys[v].k[j] + DF; b[j] = m.keys[v].k[j] - DF; }
      n1[(size_t)j * M + v] = map_find(&m, a, 0);
      n2[(size_t)j * M + v] = map_find(&m, b, 0);
    }
  }

  float* val = (float*)malloc((size_t)(M + 2) * sizeof(float));
  float* nval = (float*)malloc((size_t)(M + 2) * sizeof(float));
  const float alpha = 1.0f / (1.0f + powf(2.f, -(float)DF));
  for (int k = 0; k < K; k++) {
    const float* ip = in + (size_t)k * HW;
    float* op = out + (size_t)k * HW;
    for (int i = 0; i < M + 2; i++) val[i] = nval[i] = 0.f;
    for (int i = 0; i < HW; i++)
      for (int r = 0; r < DV; r++) val[offs[(size_t)i * DV + r] + 1] += bary[(size_t)i * DV + r] * ip[i];
    for (int j = 0; j < DV; j++) {
      if (j == skip_blur_axis) continue;
      for (int v = 0; v < M; v++) {
        float a = val[n1[(size_t)j * M + v] + 1], b = val[n2[(size_t)j * M + v] + 1];
        nval[v + 1] = val[v + 1] + 0.5f * (a + b);
      }
      float* t = val; val = nval; nval = t;
    }
    for (int i = 0; i < HW; i++) {
      float s = 0.f;
      for (int r = 0; r < DV; r++) {
        float w = bary[(size_t)i * DV + r] * alpha;
        s += w * val[offs[(size_t)i * DV + r] + 1];
      }
      op[i] = s;
    }
  }
  free(val); free(nval); free(n1); free(n2); free(offs); free(bary); free(m.slots); free(m.keys);
  return M;
}

int permuto_oracle_image(const float* image, const float* in, float* out, int K, int H, int W,
                         float sigmargb, float sigmaxy) {
  return permuto_oracle_image_variant(image, in, out, K, H, W, sigmargb, sigmaxy, -1);
}

/* Same argument order as the SWIG export bilateralfilter_batch (bilateralfilter.hpp:12). */
void permuto_oracle_batch(const float* images, int len_images, const float* ins, int len_ins, float* outs, int len_outs,
                          int N, int K, int H, int W, float sigmargb, float sigmaxy) {
  (void)len_images; (void)len_ins; (void)len_outs;
  for (int n = 0; n < N; n++)
    permuto_oracle_image(images + (size_t)n * 3 * H * W, ins + (size_t)n * K * H * W, outs + (size_t)n * K * H * W,
                         K, H, W, sigmargb, sigmaxy);
}
