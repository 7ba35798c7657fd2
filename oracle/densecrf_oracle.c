/*
 * densecrf_oracle.c -- CPU ORACLE (test infrastructure only) for the dense-CRF mean-field inference.
 *
 * A scalar restatement of densecrf 2.x (the library under pydensecrf) as the PSA-lineage crf_inference drives it
 * (DenseCRF2D, addPairwiseGaussian + addPairwiseBilateral with PottsCompatibility, DIAG_KERNEL, NORMALIZE_SYMMETRIC,
 * unary_from_softmax), written from the algorithm description.  Parity with the library itself is NOT pinned (the library
 * is not available); parity of its lattice with the reference's permutohedral.cpp is, through permuto_oracle.c: at
 * H*W % 4 == 0 (no phantom pads) densecrf_oracle_bilateral is bit-exact with permuto_oracle_batch.
 *
 * Lattice: the elevation, rank, barycentric and key steps of permuto_oracle.c with densecrf 2.x's scalar init:
 *   - every pixel is embedded alone (no phantom zero-feature pads);
 *   - rounding to the remainder-0 point: up = ceil(v)*(d+1), down = floor(v)*(d+1), rem0 = (up - e < e - down) ? up : down,
 *     so an exact tie goes to the LOWER multiple (permuto_oracle.c rounds to nearest even);
 *   - blur along axes j = 0..d, new = old + 0.5*(n1 + n2), missing neighbour 0; slice times alpha = 1/(1+2^-d).
 * CRF (per image, pixel-major internally):
 *   -U = logf(max(P, clip)); Q0 = softmax(-U) (max subtracted, expf, divided by the sequential sum);
 *   norm_k = (float)(1 / sqrt((double)L_k(1) + 1e-20)); K_k(v) = norm_k * L_k(norm_k * v);
 *   Q <- softmax(-U + compat_g * K_g(Q) + compat_b * K_b(Q)), the terms added in that order.
 * Must be compiled with -ffp-contract=off (separate multiply and add roundings, as the GPU code).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define DMAX 5

typedef struct {
  int d, n, m;                /* feature dimension, points, vertices */
  size_t cap;
  int* slots;                 /* hash slots: vertex id or -1 */
  int16_t* keys;              /* [n*(d+1)][d] by vertex id */
  int* offs;                  /* [n][d+1] vertex id of each simplex corner */
  float* bary;                /* [n][d+1] */
  int *n1, *n2;               /* [d+1][m] blur neighbours, -1 = missing */
} lattice_t;

static uint64_t key_hash(const int16_t* k, int d) {
  uint64_t r = 0;
  for (int i = 0; i < d; i++) { r += (uint64_t)(int64_t)k[i]; r *= 1664525u; }
  return r;
}

static int map_find(lattice_t* L, const int16_t* k, int create) {
  const int d = L->d;
  size_t h = key_hash(k, d) % L->cap;
  for (;;) {
    int e = L->slots[h];
    if (e < 0) {
      if (!create) return -1;
      memcpy(L->keys + (size_t)L->m * d, k, sizeof(int16_t) * d);
      L->slots[h] = L->m;
      return L->m++;
    }
    if (memcmp(L->keys + (size_t)e * d, k, sizeof(int16_t) * d) == 0) return e;
    if (++h == L->cap) h = 0;
  }
}

static void embed(const float* f, int d, int16_t keys[DMAX + 1][DMAX], float bary_out[DMAX + 1]) {
  const int dv = d + 1;
  float scale[DMAX], elevated[DMAX + 1], rem0[DMAX + 1], rank[DMAX + 1], bary[DMAX + 2];
  const float inv_std_dev = (float)(sqrt(2.0 / 3.0) * (d + 1));
  for (int i = 0; i < d; i++) scale[i] = (float)(1.0 / sqrt((double)((i + 2) * (i + 1))) * inv_std_dev);
  const float invdp1 = 1.0f / (float)dv, dp1 = (float)dv;
  float sm = 0.f;
  for (int j = d; j > 0; j--) {
    float cf = f[j - 1] * scale[j - 1];
    elevated[j] = sm - (float)j * cf;
    sm += cf;
  }
  elevated[0] = sm;
  float sum = 0.f;
  for (int i = 0; i < dv; i++) {
    float v = invdp1 * elevated[i];
    float up = ceilf(v), down = floorf(v);
    float r = (up * dp1 - elevated[i] < elevated[i] - down * dp1) ? up : down;     /* tie -> lower multiple */
    rem0[i] = r * dp1;
    sum += r;
    rank[i] = 0.f;
  }
  for (int i = 0; i < d; i++) {
    float di = elevated[i] - rem0[i];
    for (int j = i + 1; j < dv; j++) {
      float dj = elevated[j] - rem0[j];
      float c = (di < dj) ? 1.f : 0.f;
      rank[i] += c;
      rank[j] += 1.f - c;
    }
  }
  for (int i = 0; i < dv; i++) {
    rank[i] += sum;
    float add = (rank[i] < 0.f) ? dp1 : 0.f;
    float sub = (rank[i] >= dp1) ? dp1 : 0.f;
    rank[i] += add - sub;
    rem0[i] += add - sub;
  }
  for (int i = 0; i < dv + 1; i++) bary[i] = 0.f;
  for (int i = 0; i < dv; i++) {
    float v = (elevated[i] - rem0[i]) * invdp1;
    int p = d - (int)rank[i];
    bary[p] += v;
    bary[p + 1] -= v;
  }
  bary[0] += 1.0f + bary[dv];
  for (int r = 0; r < dv; r++) {
    for (int i = 0; i < d; i++) {
      int rk = (int)rank[i];
      int canon = (rk <= d - r) ? r : r - dv;
      keys[r][i] = (int16_t)(rem0[i] + (float)canon);
    }
    bary_out[r] = bary[r];
  }
}

/* feats [n][d] */
static void lattice_init(lattice_t* L, const float* feats, int n, int d) {
  const int dv = d + 1;
  L->d = d; L->n = n; L->m = 0;
  L->cap = (size_t)n * dv * 2 + 16;
  L->slots = (int*)malloc(L->cap * sizeof(int));
  memset(L->slots, 0xff, L->cap * sizeof(int));
  L->keys = (int16_t*)malloc((size_t)n * dv * d * sizeof(int16_t));
  L->offs = (int*)malloc((size_t)n * dv * sizeof(int));
  L->bary = (float*)malloc((size_t)n * dv * sizeof(float));
  for (int i = 0; i < n; i++) {
    int16_t keys[DMAX + 1][DMAX];
    float b[DMAX + 1];
    embed(feats + (size_t)i * d, d, keys, b);
    for (int r = 0; r < dv; r++) {
      L->offs[(size_t)i * dv + r] = map_find(L, keys[r], 1);
      L->bary[(size_t)i * dv + r] = b[r];
    }
  }
  const int m = L->m;
  L->n1 = (int*)malloc((size_t)m * dv * sizeof(int));
  L->n2 = (int*)malloc((size_t)m * dv * sizeof(int));
  for (int j = 0; j < dv; j++) {
    for (int v = 0; v < m; v++) {
      int16_t a[DMAX], b[DMAX];
      const int16_t* k = L->keys + (size_t)v * d;
      for (int i = 0; i < d; i++) { a[i] = k[i] - 1; b[i] = k[i] + 1; }
      if (j < d) { a[j] = k[j] + d; b[j] = k[j] - d; }
      L->n1[(size_t)j * m + v] = map_find(L, a, 0);
      L->n2[(size_t)j * m + v] = map_find(L, b, 0);
    }
  }
}

static void lattice_free(lattice_t* L) {
  free(L->slots); free(L->keys); free(L->offs); free(L->bary); free(L->n1); free(L->n2);
}

/* out[n][vs] = L(in[n][vs]): splat in pixel order, d+1 blur passes, slice.  out may alias in. */
static void lattice_compute(const lattice_t* L, const float* in, float* out, int vs) {
  const int dv = L->d + 1, m = L->m, n = L->n;
  float* val = (float*)calloc((size_t)(m + 1) * vs, sizeof(float));      /* slot 0 = missing neighbour */
  float* nval = (float*)calloc((size_t)(m + 1) * vs, sizeof(float));
  for (int i = 0; i < n; i++)
    for (int r = 0; r < dv; r++) {
      float w = L->bary[(size_t)i * dv + r];
      float* dst = val + (size_t)(L->offs[(size_t)i * dv + r] + 1) * vs;
      for (int k = 0; k < vs; k++) dst[k] += w * in[(size_t)i * vs + k];
    }
  for (int j = 0; j < dv; j++) {
    for (int v = 0; v < m; v++) {
      const float* a = val + (size_t)(L->n1[(size_t)j * m + v] + 1) * vs;
      const float* b = val + (size_t)(L->n2[(size_t)j * m + v] + 1) * vs;
      const float* o = val + (size_t)(v + 1) * vs;
      float* nv = nval + (size_t)(v + 1) * vs;
      for (int k = 0; k < vs; k++) nv[k] = o[k] + 0.5f * (a[k] + b[k]);
    }
    float* t = val; val = nval; nval = t;
  }
  const float alpha = 1.0f / (1.0f + powf(2.f, -(float)L->d));
  for (int i = 0; i < n; i++) {
    for (int k = 0; k < vs; k++) {
      float s = 0.f;
      for (int r = 0; r < dv; r++) {
        float w = L->bary[(size_t)i * dv + r] * alpha;
        s += w * val[(size_t)(L->offs[(size_t)i * dv + r] + 1) * vs + k];
      }
      out[(size_t)i * vs + k] = s;
    }
  }
  free(val); free(nval);
}

/* features of the two kernels of DenseCRF2D: x is the column, y the row; image [3][H][W] */
static float* features(const float* image, int H, int W, int d, float sxy, float srgb) {
  const int n = H * W;
  float* f = (float*)malloc((size_t)n * d * sizeof(float));
  for (int i = 0; i < n; i++) {
    f[(size_t)i * d + 0] = (float)(i % W) / sxy;
    f[(size_t)i * d + 1] = (float)(i / W) / sxy;
    for (int c = 2; c < d; c++) f[(size_t)i * d + c] = image[(size_t)(c - 2) * n + i] / srgb;
  }
  return f;
}

static void softmax(const float* t, float* q, int C) {
  float m = -INFINITY, s = 0.f;
  for (int k = 0; k < C; k++) m = fmaxf(m, t[k]);
  for (int k = 0; k < C; k++) { q[k] = expf(t[k] - m); s += q[k]; }
  for (int k = 0; k < C; k++) q[k] = q[k] / s;
}

/* The bilateral lattice filter alone, planes [K][H][W] in and out (the layout of permuto_oracle_batch); returns M. */
int densecrf_oracle_bilateral(const float* image, const float* in, float* out, int K, int H, int W, float srgb, float sxy) {
  const int n = H * W;
  float* f = features(image, H, W, 5, sxy, srgb);
  lattice_t L;
  lattice_init(&L, f, n, 5);
  float* buf = (float*)malloc((size_t)n * K * sizeof(float));
  for (int k = 0; k < K; k++)
    for (int i = 0; i < n; i++) buf[(size_t)i * K + k] = in[(size_t)k * n + i];
  lattice_compute(&L, buf, buf, K);
  for (int k = 0; k < K; k++)
    for (int i = 0; i < n; i++) out[(size_t)k * n + i] = buf[(size_t)i * K + k];
  const int m = L.m;
  lattice_free(&L); free(f); free(buf);
  return m;
}

static void pairwise(const lattice_t* L, const float* norm, const float* Q, float* out, int n, int C) {
  for (int i = 0; i < n; i++)
    for (int k = 0; k < C; k++) out[(size_t)i * C + k] = norm[i] * Q[(size_t)i * C + k];
  lattice_compute(L, out, out, C);
  for (int i = 0; i < n; i++)
    for (int k = 0; k < C; k++) out[(size_t)i * C + k] = norm[i] * out[(size_t)i * C + k];
}

/* One image: image [3][H][W] in 0..255, probs and q [C][H][W].  lattice_sizes (nullable) receives {M_gauss, M_bilateral}. */
void densecrf_oracle(const float* image, const float* probs, float* q, int C, int H, int W, int n_iter, float sxy_g,
                     float compat_g, float sxy_b, float srgb, float compat_b, float clip, int* lattice_sizes) {
  const int n = H * W;
  float* fg = features(image, H, W, 2, sxy_g, 1.f);
  float* fb = features(image, H, W, 5, sxy_b, srgb);
  lattice_t Lg, Lb;
  lattice_init(&Lg, fg, n, 2);
  lattice_init(&Lb, fb, n, 5);
  if (lattice_sizes) { lattice_sizes[0] = Lg.m; lattice_sizes[1] = Lb.m; }
  float* ng = (float*)malloc((size_t)n * sizeof(float));
  float* nb = (float*)malloc((size_t)n * sizeof(float));
  float* ones = (float*)malloc((size_t)n * sizeof(float));
  for (int i = 0; i < n; i++) ones[i] = 1.f;
  lattice_compute(&Lg, ones, ng, 1);
  lattice_compute(&Lb, ones, nb, 1);
  for (int i = 0; i < n; i++) {
    ng[i] = (float)(1.0 / sqrt((double)ng[i] + 1e-20));
    nb[i] = (float)(1.0 / sqrt((double)nb[i] + 1e-20));
  }
  float* mu = (float*)malloc((size_t)n * C * sizeof(float));      /* -U, pixel-major */
  float* Q = (float*)malloc((size_t)n * C * sizeof(float));
  float* kg = (float*)malloc((size_t)n * C * sizeof(float));
  float* kb = (float*)malloc((size_t)n * C * sizeof(float));
  float* t = (float*)malloc((size_t)C * sizeof(float));
  for (int i = 0; i < n; i++)
    for (int k = 0; k < C; k++) mu[(size_t)i * C + k] = logf(fmaxf(probs[(size_t)k * n + i], clip));
  for (int i = 0; i < n; i++) softmax(mu + (size_t)i * C, Q + (size_t)i * C, C);
  for (int it = 0; it < n_iter; it++) {
    pairwise(&Lg, ng, Q, kg, n, C);
    pairwise(&Lb, nb, Q, kb, n, C);
    for (int i = 0; i < n; i++) {
      for (int k = 0; k < C; k++) {
        size_t e = (size_t)i * C + k;
        t[k] = mu[e] + compat_g * kg[e];
        t[k] = t[k] + compat_b * kb[e];
      }
      softmax(t, Q + (size_t)i * C, C);
    }
  }
  for (int k = 0; k < C; k++)
    for (int i = 0; i < n; i++) q[(size_t)k * n + i] = Q[(size_t)i * C + k];
  lattice_free(&Lg); lattice_free(&Lb);
  free(fg); free(fb); free(ng); free(nb); free(ones); free(mu); free(Q); free(kg); free(kb); free(t);
}
