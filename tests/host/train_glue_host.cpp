// Host run of the training-glue phases (hold_b200/csrc/train_glue_phases.h), block by block, thread by thread.
#include <vector>

#include "../../hold_b200/csrc/train_glue_phases.h"

using namespace hold::glue;

// frame-major points [B, P]; tfs [B,16,4,4] (hand) / [B,4,4] (object)
extern "C" int nd_fwd_host(int hand, int B, int P, const float* xc, const float* g, const float* sdf, const float* tfs, const float* cano,
                           const float* skin_w, float beta, float* normal, float* density, float* stash) {
  const int ld = hand ? kStashHand : kStashObj;
  for (int b = 0; b < B; ++b) {
    float Ji[9];
    if (!hand) inv3(tfs + b * 16, 4, Ji);
    for (int p = 0; p < P; ++p) {
      const size_t gp = (size_t)b * P + p;
      float* st = stash + gp * ld;
      if (hand) hand_stash(xc + 3 * gp, cano, skin_w, tfs + (size_t)b * 256, st);
      else
        for (int e = 0; e < 9; ++e) st[e] = Ji[e];
      nd_point_fwd(st, g + 3 * gp, sdf[gp], beta, normal + 3 * gp, density + gp);
    }
  }
  return 0;
}

extern "C" int nd_bwd_host(int hand, int nt, int B, int P, const float* g, const float* sdf, float beta, const float* stash,
                           const float* d_normal, const float* d_density, float* d_g, float* d_sdf, float* d_tfs, float* d_beta) {
  const int nb = P > 0 ? (P + nt - 1) / nt : 1, npart = hand ? kPartHand : kPartObj, ld = hand ? kStashHand : kStashObj;
  std::vector<float> scr(scratch_floats(hand, nt)), partials((size_t)B * nb * npart);
  for (int b = 0; b < B; ++b) {
    const size_t o = (size_t)b * P;
    for (int blk = 0; blk < nb; ++blk) {
      for (int t = 0; t < nt; ++t)
        nd_bwd_p0(hand, t, nt, blk * nt + t, P, stash + o * ld, g + o * 3, sdf + o, beta, d_normal ? d_normal + o * 3 : nullptr,
                  d_density ? d_density + o : nullptr, d_g + o * 3, d_sdf + o, scr.data());
      for (int t = 0; t < nt; ++t) nd_bwd_p1(hand, t, nt, scr.data(), partials.data() + ((size_t)b * nb + blk) * npart);
    }
  }
  const int per = hand ? 256 : 16;
  for (int b = 0; b < B; ++b)
    for (int e = 0; e < per; ++e) nd_bwd_final_tfs(hand, e, nb, partials.data() + (size_t)b * nb * npart, d_tfs + (size_t)b * per);
  *d_beta = nd_bwd_final_beta(hand, B * nb, partials.data());
  return 0;
}

// R rays; z [32]; sdf at sdf[(r*32 + k) * ld]
extern "C" int bg_fwd_host(int R, const float* z, const float* sdf, int ld, const float* rgb, const float* fgw, float* bg_rgb,
                           float* only, float* sem) {
  for (int r = 0; r < R; ++r) {
    bg_integrate_fwd(z, sdf + (size_t)r * kBgN * ld, ld, rgb + (size_t)r * kBgN * 3, only + 3 * r);
    for (int c = 0; c < 3; ++c) bg_rgb[3 * r + c] = fgw[r] * only[3 * r + c];
    sem[4 * r] = fgw[r], sem[4 * r + 1] = sem[4 * r + 2] = sem[4 * r + 3] = 0.f;
  }
  return 0;
}

extern "C" int bg_bwd_host(int R, const float* z, const float* sdf, int ld, const float* rgb, const float* fgw, const float* g_rgb,
                           const float* g_only, const float* g_sem, float* d_rgb, float* d_sdf, float* d_fgw) {
  for (int r = 0; r < R; ++r) {
    const size_t s0 = (size_t)r * kBgN;
    bg_integrate_bwd(z, sdf + s0 * ld, ld, rgb + s0 * 3, fgw[r], g_rgb ? g_rgb + 3 * r : nullptr, g_only ? g_only + 3 * r : nullptr,
                     g_sem ? g_sem + 4 * r : nullptr, d_rgb + s0 * 3, d_sdf + s0, d_fgw + r);
  }
  return 0;
}
