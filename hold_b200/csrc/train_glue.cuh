// Kernels of the training-mode glue (arithmetic in train_glue_phases.h):
//  * k_nd_fwd / k_nd_bwd / k_nd_bwd_final: normal + Laplace density of the node's samples and their reverse mode.  Points are
//    frame-major [B, P]; a block holds 128 points of one frame (blockIdx.y) with the frame's transforms (and, hand, the canonical
//    vertices) in shared memory.  The backward writes per-block partials; the final kernel adds them in block order (deterministic).
//  * k_bg_inputs: the background's point and view-direction embeddings of the 32 inverse-sphere samples per ray.
//  * k_bg_integrate / k_bg_integrate_bwd: the AbsDensity integration of the 32 samples, one ray per thread.
#pragma once
#include "common.cuh"
#include "background.cuh"
#include "train_glue_phases.h"

namespace hold {

constexpr int kGlueThreads = 128;

template <bool HAND>
__global__ void __launch_bounds__(kGlueThreads)
k_nd_fwd(int P, const float* __restrict__ xc, const float* __restrict__ grad, const float* __restrict__ sdf,
         const float* __restrict__ tfs, const float* __restrict__ cano, const float* __restrict__ skin_w,
         const float* __restrict__ beta, float* __restrict__ normal, float* __restrict__ density, float* __restrict__ stash) {
  __shared__ float sv[HAND ? kVerts * 3 : 1];
  __shared__ float stf[HAND ? kJoints * 16 : 16];
  __shared__ float sJi[9];
  const int b = blockIdx.y;
  if (HAND) {
    for (int t = threadIdx.x; t < kVerts * 3; t += blockDim.x) sv[t] = cano[t];
    for (int t = threadIdx.x; t < kJoints * 16; t += blockDim.x) stf[t] = tfs[(size_t)b * kJoints * 16 + t];
  } else {
    if (threadIdx.x < 16) stf[threadIdx.x] = tfs[b * 16 + threadIdx.x];
    __syncthreads();
    if (threadIdx.x == 0) glue::inv3(stf, 4, sJi);
  }
  __syncthreads();
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  const size_t gp = (size_t)b * P + p;
  float st[HAND ? glue::kStashHand : glue::kStashObj];
  if (HAND) {
    const float x[3] = {xc[3 * gp], xc[3 * gp + 1], xc[3 * gp + 2]};
    glue::hand_stash(x, sv, skin_w, stf, st);
  } else {
#pragma unroll
    for (int e = 0; e < 9; ++e) st[e] = sJi[e];
  }
  const float g[3] = {grad[3 * gp], grad[3 * gp + 1], grad[3 * gp + 2]};
  float n[3], rho;
  glue::nd_point_fwd(st, g, sdf[gp], beta[0], n, &rho);
  normal[3 * gp] = n[0], normal[3 * gp + 1] = n[1], normal[3 * gp + 2] = n[2];
  density[gp] = rho;
  constexpr int ld = HAND ? glue::kStashHand : glue::kStashObj;
#pragma unroll
  for (int e = 0; e < ld; ++e) stash[gp * ld + e] = st[e];
}

template <bool HAND>
__global__ void __launch_bounds__(kGlueThreads)
k_nd_bwd(int P, const float* __restrict__ grad, const float* __restrict__ sdf, const float* __restrict__ beta,
         const float* __restrict__ stash, const float* __restrict__ d_normal, const float* __restrict__ d_density,
         float* __restrict__ d_grad, float* __restrict__ d_sdf, float* __restrict__ partials) {
  constexpr int kScr = kGlueThreads * ((HAND ? glue::kJ : 0) + 10);
  constexpr int kPart = HAND ? glue::kPartHand : glue::kPartObj;
  constexpr int ld = HAND ? glue::kStashHand : glue::kStashObj;
  __shared__ float scr[kScr];
  const int b = blockIdx.y, tid = threadIdx.x, nt = blockDim.x;
  const size_t o = (size_t)b * P;
  glue::nd_bwd_p0(HAND, tid, nt, blockIdx.x * nt + tid, P, stash + o * ld, grad + o * 3, sdf + o, beta[0],
                  d_normal ? d_normal + o * 3 : nullptr, d_density ? d_density + o : nullptr, d_grad + o * 3, d_sdf + o, scr);
  __syncthreads();
  glue::nd_bwd_p1(HAND, tid, nt, scr, partials + ((size_t)b * gridDim.x + blockIdx.x) * kPart);
}

// grid B blocks x (hand 256 | object 16) threads; block 0, thread 0 also reduces d beta over all B * n_blocks partials
template <bool HAND>
__global__ void k_nd_bwd_final(int n_blocks, const float* __restrict__ partials, float* __restrict__ d_tfs, float* __restrict__ d_beta) {
  constexpr int kPart = HAND ? glue::kPartHand : glue::kPartObj;
  const int b = blockIdx.x, o = threadIdx.x;
  glue::nd_bwd_final_tfs(HAND, o, n_blocks, partials + (size_t)b * n_blocks * kPart, d_tfs + (size_t)b * (HAND ? 256 : 16));
  if (b == 0 && o == 0) d_beta[0] = glue::nd_bwd_final_beta(HAND, gridDim.x * n_blocks, partials);
}

// one thread per (ray, sample): emb_pts [R*32, 84] = PE-10 of depth2pts_outside, emb_view [R*32, 27] = PE-4 of the ray direction
__global__ void __launch_bounds__(kGlueThreads)
k_bg_inputs(int R, float r_sphere, const float* __restrict__ cam, const float* __restrict__ dirs, float* __restrict__ emb_pts,
            float* __restrict__ emb_view) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= R * kBgN) return;
  const int ray = i / kBgN, k = i - ray * kBgN;
  const float o[3] = {cam[3 * ray], cam[3 * ray + 1], cam[3 * ray + 2]};
  const float d[3] = {dirs[3 * ray], dirs[3 * ray + 1], dirs[3 * ray + 2]};
  float p4[4];
  depth2pts_outside(o, d, bg_depth(k, r_sphere), r_sphere, p4);
  embed_generic<4, 10>(p4, emb_pts + (size_t)i * kBgEmbed);
  embed_generic<3, 4>(d, emb_view + (size_t)i * kBgView);
}

__global__ void __launch_bounds__(kGlueThreads)
k_bg_integrate(int R, float r_sphere, const float* __restrict__ sdf, int ld, const float* __restrict__ rgb,
               const float* __restrict__ fg_bg_weights, float* __restrict__ bg_rgb, float* __restrict__ bg_rgb_only,
               float* __restrict__ bg_sem) {
  __shared__ float sz[kBgN];
  if (threadIdx.x < kBgN) sz[threadIdx.x] = bg_depth(threadIdx.x, r_sphere);
  __syncthreads();
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= R) return;
  float only[3];
  glue::bg_integrate_fwd(sz, sdf + (size_t)r * kBgN * ld, ld, rgb + (size_t)r * kBgN * 3, only);
  const float wbg = fg_bg_weights[r];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    if (bg_rgb_only) bg_rgb_only[3 * r + c] = only[c];
    if (bg_rgb) bg_rgb[3 * r + c] = wbg * only[c];
  }
  if (bg_sem) { bg_sem[4 * r] = wbg; bg_sem[4 * r + 1] = 0.f; bg_sem[4 * r + 2] = 0.f; bg_sem[4 * r + 3] = 0.f; }
}

__global__ void __launch_bounds__(kGlueThreads)
k_bg_integrate_bwd(int R, float r_sphere, const float* __restrict__ sdf, int ld, const float* __restrict__ rgb,
                   const float* __restrict__ fg_bg_weights, const float* __restrict__ g_rgb, const float* __restrict__ g_only,
                   const float* __restrict__ g_sem, float* __restrict__ d_rgb, float* __restrict__ d_sdf, float* __restrict__ d_fgw) {
  __shared__ float sz[kBgN];
  if (threadIdx.x < kBgN) sz[threadIdx.x] = bg_depth(threadIdx.x, r_sphere);
  __syncthreads();
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= R) return;
  const size_t s0 = (size_t)r * kBgN;
  glue::bg_integrate_bwd(sz, sdf + s0 * ld, ld, rgb + s0 * 3, fg_bg_weights[r], g_rgb ? g_rgb + 3 * r : nullptr,
                         g_only ? g_only + 3 * r : nullptr, g_sem ? g_sem + 4 * r : nullptr, d_rgb + s0 * 3, d_sdf + s0, d_fgw + r);
}

}  // namespace hold
