// Per-point glue of the training forward and its reverse mode (hold_b200/train.py NormalDensityFn, BgIntegrateFn):
//  * the normal of extract_features (engine/volsdf_utils.py:66-102) with DETACHED skinning weights (mano/deformer.py:101):
//      J = sum_j w_j tfs_j[:3,:3] (hand; w from the 15 nearest CANONICAL vertices) or tfs[:3,:3] (object),
//      m = g . J^-1 (row vector),  n = m / max(|m|, 1e-6)
//    and the Laplace density rho(s, beta) of engine/density.py:21-26;
//  * the AbsDensity integration of the background's 32 inverse-sphere samples (background.py:137-165).
// Reverse mode of the normal:  d_m = d_n / |m| - m (m . d_n) / |m|^3  (d_n / eps when |m| <= eps),  d_g = J^-1 d_m,
// d_J^-1 = g (x) d_m,  d_J = -J^-T d_J^-1 J^-T = -m (x) d_g.
// Written as per-thread phases (host-executable, tests/host/train_glue_host.cpp); every sum over points is fixed-order: per-block
// partials, then one pass over the blocks in order.
#pragma once
#include <math.h>

#if defined(__CUDACC__)
#define HOLD_HD __host__ __device__ __forceinline__
#else
#ifndef HOLD_HD
#define HOLD_HD inline
#endif
#endif

#if defined(__CUDA_ARCH__)
#define HOLD_GLUE_UNROLL _Pragma("unroll")
#else
#define HOLD_GLUE_UNROLL
#endif

namespace hold {
namespace glue {

constexpr int kK = 15, kJ = 16, kV = 778;
constexpr int kStashHand = 9 + kJ;      // per point: J^-1 (row-major) | the 16 blended skinning weights
constexpr int kStashObj = 9;            // per point: J^-1
constexpr int kPartHand = kJ * 9 + 1;   // per block: sum_p w_pj d_J_p (16 x 9) | d beta
constexpr int kPartObj = 9 + 1;         // per block: sum_p d_J_p | d beta
constexpr int kBgN = 32;                // background samples per ray
constexpr float kNormEps = 1e-6f;       // F.normalize eps

// products and sums without FMA contraction on the device: the neighbour selection must agree with the other KNN kernels
HOLD_HD float mul_rn(float a, float b) {
#if defined(__CUDA_ARCH__)
  return __fmul_rn(a, b);
#else
  return a * b;
#endif
}
HOLD_HD float add_rn(float a, float b) {
#if defined(__CUDA_ARCH__)
  return __fadd_rn(a, b);
#else
  return a + b;
#endif
}

// exact 15 nearest of the 778 vertices: ascending squared distance, ties -> lower index (geom.cuh knn15)
HOLD_HD void knn15(const float* v /*[778,3]*/, float px, float py, float pz, float* d /*15*/, int* idx /*15*/) {
  for (int k = 0; k < kK; ++k) { d[k] = 3.0e38f; idx[k] = 0; }
  for (int i = 0; i < kV; ++i) {
    const float dx = px - v[3 * i], dy = py - v[3 * i + 1], dz = pz - v[3 * i + 2];
    const float dist = add_rn(add_rn(mul_rn(dx, dx), mul_rn(dy, dy)), mul_rn(dz, dz));
    if (dist < d[kK - 1]) {
      d[kK - 1] = dist;
      idx[kK - 1] = i;
      HOLD_GLUE_UNROLL
      for (int k = kK - 1; k > 0; --k) {
        if (d[k] < d[k - 1]) {
          const float td = d[k]; d[k] = d[k - 1]; d[k - 1] = td;
          const int ti = idx[k]; idx[k] = idx[k - 1]; idx[k - 1] = ti;
        }
      }
    }
  }
}

// query_skinning_weights_multi (deformer.py:84-105): conf = softmax(-min(d^2, 4)) over the 15 neighbours, w = sum conf . W
HOLD_HD void skin_weights(const float* d, const int* idx, const float* skin_w /*[778,16]*/, float* w /*16*/) {
  float conf[kK], csum = 0.f;
  HOLD_GLUE_UNROLL
  for (int k = 0; k < kK; ++k) {
    conf[k] = expf(-fminf(d[k], 4.0f));
    csum += conf[k];
  }
  HOLD_GLUE_UNROLL
  for (int j = 0; j < kJ; ++j) w[j] = 0.f;
  HOLD_GLUE_UNROLL
  for (int k = 0; k < kK; ++k) {
    const float c = conf[k] / csum;
    HOLD_GLUE_UNROLL
    for (int j = 0; j < kJ; ++j) w[j] += skin_w[idx[k] * kJ + j] * c;
  }
}

HOLD_HD bool inv3(const float* A /*row-major 3x3, row stride rs*/, int rs, float* Ai /*9*/) {
  const float a = A[0], b = A[1], c = A[2], d = A[rs], e = A[rs + 1], f = A[rs + 2], g = A[2 * rs], h = A[2 * rs + 1],
              i = A[2 * rs + 2];
  const float c0 = e * i - f * h, c1 = f * g - d * i, c2 = d * h - e * g;
  const float id = 1.0f / (a * c0 + b * c1 + c * c2);
  Ai[0] = c0 * id, Ai[1] = (c * h - b * i) * id, Ai[2] = (b * f - c * e) * id;
  Ai[3] = c1 * id, Ai[4] = (a * i - c * g) * id, Ai[5] = (c * d - a * f) * id;
  Ai[6] = c2 * id, Ai[7] = (b * g - a * h) * id, Ai[8] = (a * e - b * d) * id;
  return isfinite(id);
}

HOLD_HD float laplace(float s, float beta) {
  const float sg = (s > 0.f) ? 1.f : ((s < 0.f) ? -1.f : 0.f);
  return (1.0f / beta) * (0.5f + 0.5f * sg * expm1f(-fabsf(s) / beta));
}

// ---------------------------------------------------------------------------------------------- normal + density, forward
// hand: the stash row is [J^-1 (9) | w (16)] of the point x_c; tfs [16,16] of its frame
HOLD_HD void hand_stash(const float* xc, const float* cano /*[778,3]*/, const float* skin_w, const float* tfs, float* stash) {
  float d[kK];
  int idx[kK];
  knn15(cano, xc[0], xc[1], xc[2], d, idx);
  float* w = stash + 9;
  skin_weights(d, idx, skin_w, w);
  float J[9];
  HOLD_GLUE_UNROLL
  for (int e = 0; e < 9; ++e) J[e] = 0.f;
  HOLD_GLUE_UNROLL
  for (int j = 0; j < kJ; ++j) {
    HOLD_GLUE_UNROLL
    for (int r = 0; r < 3; ++r) {
      HOLD_GLUE_UNROLL
      for (int c = 0; c < 3; ++c) J[3 * r + c] += w[j] * tfs[j * 16 + 4 * r + c];
    }
  }
  inv3(J, 3, stash);
}

// m = g . J^-1
HOLD_HD void row_times(const float* g, const float* Ji, float* m) {
  HOLD_GLUE_UNROLL
  for (int c = 0; c < 3; ++c) m[c] = g[0] * Ji[c] + g[1] * Ji[3 + c] + g[2] * Ji[6 + c];
}

// normal (3) and density of one point from its J^-1; density skipped when rho is NULL
HOLD_HD void nd_point_fwd(const float* Ji, const float* g, float s, float beta, float* n, float* rho) {
  float m[3];
  row_times(g, Ji, m);
  const float nm = fmaxf(sqrtf(m[0] * m[0] + m[1] * m[1] + m[2] * m[2]), kNormEps);
  n[0] = m[0] / nm, n[1] = m[1] / nm, n[2] = m[2] / nm;
  if (rho != nullptr) *rho = laplace(s, beta);
}

// ---------------------------------------------------------------------------------------------- normal + density, reverse
// one point: seeds dn (3, or NULL) and drho -> d_g (3), d_J (9), d_sdf, d_beta
HOLD_HD void nd_point_bwd(const float* Ji, const float* g, float s, float beta, const float* dn, float drho, float* dg,
                          float* dJ, float* ds, float* dbeta) {
  float m[3], dm[3] = {0.f, 0.f, 0.f};
  row_times(g, Ji, m);
  if (dn != nullptr) {
    const float nm = sqrtf(m[0] * m[0] + m[1] * m[1] + m[2] * m[2]);
    if (nm > kNormEps) {
      const float md = (m[0] * dn[0] + m[1] * dn[1] + m[2] * dn[2]) / (nm * nm * nm);
      HOLD_GLUE_UNROLL
      for (int c = 0; c < 3; ++c) dm[c] = dn[c] / nm - m[c] * md;
    } else {
      HOLD_GLUE_UNROLL
      for (int c = 0; c < 3; ++c) dm[c] = dn[c] / kNormEps;
    }
  }
  HOLD_GLUE_UNROLL
  for (int r = 0; r < 3; ++r) dg[r] = Ji[3 * r] * dm[0] + Ji[3 * r + 1] * dm[1] + Ji[3 * r + 2] * dm[2];
  HOLD_GLUE_UNROLL
  for (int r = 0; r < 3; ++r) {
    HOLD_GLUE_UNROLL
    for (int c = 0; c < 3; ++c) dJ[3 * r + c] = -m[r] * dg[c];
  }
  // torch's sign / abs have zero derivative at 0: d_sdf is exactly 0 there
  const float a = fabsf(s), e = expf(-a / beta), sg = (s > 0.f) ? 1.f : ((s < 0.f) ? -1.f : 0.f);
  *ds = (s == 0.f) ? 0.f : -drho * e / (2.f * beta * beta);
  *dbeta = drho * (-laplace(s, beta) / beta + 0.5f * sg * e * a / (beta * beta * beta));
}

// scratch of one block of nt points: hand w [nt][16] | q [nt][10]; object q [nt][10]; q = d_J (9) | d beta
HOLD_HD int scratch_floats(bool hand, int nt) { return nt * ((hand ? kJ : 0) + 10); }

// P0: thread = point p (or idle).  stash: the forward's row of the point; dn / drho / d_g / d_sdf indexed by p (seeds may be NULL).
HOLD_HD void nd_bwd_p0(bool hand, int tid, int nt, int p, int P, const float* stash, const float* g, const float* sdf, float beta,
                       const float* dn, const float* drho, float* d_g, float* d_sdf, float* scr) {
  float* w = scr + tid * kJ;
  float* q = scr + (hand ? nt * kJ : 0) + tid * 10;
  if (p >= P) {
    if (hand)
      for (int j = 0; j < kJ; ++j) w[j] = 0.f;
    for (int e = 0; e < 10; ++e) q[e] = 0.f;
    return;
  }
  const int ld = hand ? kStashHand : kStashObj;
  const float* st = stash + (size_t)ld * p;
  float dg[3], ds;
  nd_point_bwd(st, g + 3 * p, sdf[p], beta, dn ? dn + 3 * p : nullptr, drho ? drho[p] : 0.f, dg, q, &ds, q + 9);
  d_g[3 * p] = dg[0], d_g[3 * p + 1] = dg[1], d_g[3 * p + 2] = dg[2];
  d_sdf[p] = ds;
  if (hand)
    for (int j = 0; j < kJ; ++j) w[j] = st[9 + j];
}

// P1: thread o < kPart*: this block's partial sums over its nt points
HOLD_HD void nd_bwd_p1(bool hand, int tid, int nt, const float* scr, float* partial) {
  const float* q = scr + (hand ? nt * kJ : 0);
  const int n = hand ? kPartHand : kPartObj;
  for (int o = tid; o < n; o += nt) {
    float acc = 0.f;
    if (hand && o < kJ * 9) {
      const int j = o / 9, e = o % 9;
      for (int p = 0; p < nt; ++p) acc += scr[p * kJ + j] * q[p * 10 + e];
    } else {
      const int e = hand ? 9 : o;
      for (int p = 0; p < nt; ++p) acc += q[p * 10 + e];
    }
    partial[o] = acc;
  }
}

// final, transforms: entry o of one frame's d_tfs (hand: o < 256 over [16,4,4]; object: o < 16 over [4,4]) = sum over the frame's
// n_blocks partials in order; only the 3x3 blocks carry gradient
HOLD_HD void nd_bwd_final_tfs(bool hand, int o, int n_blocks, const float* partials /*[n_blocks][kPart*] of the frame*/, float* d_tfs) {
  const int j = o / 16, e = o % 16, r = e / 4, c = e % 4;
  const int n = hand ? kPartHand : kPartObj;
  float acc = 0.f;
  if (r < 3 && c < 3) {
    const int pe = (hand ? j * 9 : 0) + 3 * r + c;
    for (int b = 0; b < n_blocks; ++b) acc += partials[(size_t)b * n + pe];
  }
  d_tfs[o] = acc;
}

// final, beta: sum over all blocks of all frames, in order
HOLD_HD float nd_bwd_final_beta(bool hand, int total_blocks, const float* partials) {
  const int n = hand ? kPartHand : kPartObj;
  float acc = 0.f;
  for (int b = 0; b < total_blocks; ++b) acc += partials[(size_t)b * n + n - 1];
  return acc;
}

// ---------------------------------------------------------------------------------------------- background integration
// One ray: z [32] the flipped inverse-sphere depths (1/R_s ... 0), sdf column with stride ld, rgb [32,3].
// dens = |sdf|, dists = z_k - z_{k+1} (last 1e10), w_k = (1 - e^-fe_k) e^-sum_{i<k} fe_i.
HOLD_HD float bg_dist(const float* z, int k) { return (k + 1 < kBgN) ? z[k] - z[k + 1] : 1.0e10f; }

HOLD_HD void bg_integrate_fwd(const float* z, const float* sdf, int ld, const float* rgb, float* only /*3*/) {
  float cum = 0.f, acc[3] = {0.f, 0.f, 0.f};
  HOLD_GLUE_UNROLL
  for (int k = 0; k < kBgN; ++k) {
    const float fe = bg_dist(z, k) * fabsf(sdf[(size_t)k * ld]);
    const float w = (1.0f - expf(-fe)) * expf(-cum);
    cum += fe;
    acc[0] += w * rgb[3 * k], acc[1] += w * rgb[3 * k + 1], acc[2] += w * rgb[3 * k + 2];
  }
  only[0] = acc[0], only[1] = acc[1], only[2] = acc[2];
}

// seeds (each may be NULL = 0): g_rgb (3) of bg_rgb = fgw . only, g_only (3), g_sem (4) of bg_semantics = fgw . [1,0,0,0]
// -> d_rgb [32,3], d_sdf [32] (contiguous), d_fgw.
// With a_k = dL/dw_k = rgb_k . go:  dL/dfe_k = a_k e^-fe_k T_k - sum_{j>k} a_j w_j.  Both terms are ~ a T_{k+1} and nearly cancel when
// the colour varies little along the ray (the last sample, dists 1e10, takes the rest of the transmittance), so it is evaluated
// through T_{k+1} = sum_{j>k} w_j + T_end (the w_j telescope) as  sum_{j>k} (a_k - a_j) w_j + a_k T_end,  with a_k - a_j formed
// from the colour differences: no cancellation, float32 stays at its own precision.
HOLD_HD void bg_integrate_bwd(const float* z, const float* sdf, int ld, const float* rgb, float fgw, const float* g_rgb,
                              const float* g_only, const float* g_sem, float* d_rgb, float* d_sdf, float* d_fgw) {
  float go[3];
  for (int c = 0; c < 3; ++c) go[c] = (g_only ? g_only[c] : 0.f) + (g_rgb ? fgw * g_rgb[c] : 0.f);
  float w[kBgN], cum = 0.f, only[3] = {0.f, 0.f, 0.f};
  HOLD_GLUE_UNROLL
  for (int k = 0; k < kBgN; ++k) {
    const float fe = bg_dist(z, k) * fabsf(sdf[(size_t)k * ld]);
    w[k] = (1.0f - expf(-fe)) * expf(-cum);
    cum += fe;
    const float* c = rgb + 3 * k;
    only[0] += w[k] * c[0], only[1] += w[k] * c[1], only[2] += w[k] * c[2];
    d_rgb[3 * k] = w[k] * go[0], d_rgb[3 * k + 1] = w[k] * go[1], d_rgb[3 * k + 2] = w[k] * go[2];
  }
  const float t_end = expf(-cum);
  HOLD_GLUE_UNROLL
  for (int k = 0; k < kBgN; ++k) {
    const float* c = rgb + 3 * k;
    float dfe = (c[0] * go[0] + c[1] * go[1] + c[2] * go[2]) * t_end;
    for (int j = k + 1; j < kBgN; ++j) {
      const float* cj = rgb + 3 * j;
      dfe += ((c[0] - cj[0]) * go[0] + (c[1] - cj[1]) * go[1] + (c[2] - cj[2]) * go[2]) * w[j];
    }
    const float s = sdf[(size_t)k * ld];
    const float sg = (s > 0.f) ? 1.f : ((s < 0.f) ? -1.f : 0.f);
    d_sdf[k] = dfe * bg_dist(z, k) * sg;
  }
  float dw = g_sem ? g_sem[0] : 0.f;
  if (g_rgb) dw += g_rgb[0] * only[0] + g_rgb[1] * only[1] + g_rgb[2] * only[2];
  *d_fgw = dw;
}

}  // namespace glue
}  // namespace hold
