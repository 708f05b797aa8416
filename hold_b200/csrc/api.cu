// C ABI of hold_b200 (include/hold_b200.h): context, weight packing, launch sequences.  Host-side logic
// only — every arithmetic step of the path lives in the kernels included below.
#include <stdarg.h>
#include <stdlib.h>
#include <new>
#include <algorithm>

#include "common.cuh"
#include "geom.cuh"
#include "sampler.cuh"
#include "mlp_simt.cuh"
#include "mlp_tc.cuh"
#include "composite.cuh"
#include "background.cuh"
#include "background_tc.cuh"
#include "pose_bwd.cuh"
#include "mesh_sdf.cuh"
#include "mise.cuh"
#include "mc.cuh"
#include "warp_bwd.cuh"
#include "train.cuh"
#include "wgrad_tc.cuh"
#include "train_glue.cuh"

namespace hold {

static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

enum WsSlot { WS_Z = 0, WS_SDF, WS_ZNEW, WS_SDFNEW, WS_BETA, WS_FAR, WS_XC, WS_SSDF, WS_GRAD, WS_FEAT, WS_PE, WS_ZTMP, WS_SIG, WS_BGSDF, WS_BGFEAT, WS_BGRGB, WS_COUNT };

int ws_get(hold_ctx* ctx, int slot, size_t bytes, void** out) {
  Buffer& b = ctx->ws[slot];
  if (b.bytes < bytes) {
    if (b.p) HOLD_CUDA(cudaFree(b.p));
    b.p = nullptr, b.bytes = 0;
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&b.p, want);
    if (e != cudaSuccess) {
      set_error("workspace allocation of %zu bytes failed: %s", want, cudaGetErrorString(e));
      return HOLD_E_NOMEM;
    }
    b.bytes = want;
  }
  *out = b.p;
  return HOLD_OK;
}
#define WS(slot, type, count, var)                                                     \
  type* var = nullptr;                                                                 \
  {                                                                                    \
    void* _p;                                                                          \
    int _rc = ws_get(ctx, slot, sizeof(type) * (size_t)(count), &_p);                  \
    if (_rc) return _rc;                                                               \
    var = (type*)_p;                                                                   \
  }

static int dev_alloc(float** p, size_t n) {
  if (*p) return HOLD_OK;
  HOLD_CUDA(cudaMalloc((void**)p, n * sizeof(float)));
  return HOLD_OK;
}

static int check_node(hold_ctx* ctx, int node, bool need_weights) {
  HOLD_REQUIRE(ctx != nullptr, "ctx is NULL");
  HOLD_REQUIRE(node >= 0 && node < HOLD_MAX_NODES, "node %d out of range", node);
  if (!ctx->nodes[node].configured) { set_error("node %d not configured", node); return HOLD_E_STATE; }
  if (need_weights && !ctx->nodes[node].has_weights) { set_error("node %d has no weights", node); return HOLD_E_STATE; }
  HOLD_CUDA(cudaSetDevice(ctx->device));   // launches go to the context's device whatever the caller's current device is
  return HOLD_OK;
}

// ------------------------------------------------------------------------------------------------ MLP launches
static int fill_sdf_args(const NodeState& ns, SimtArgs& a, bool jvp) {
  a.n_layers = jvp ? 9 : 8;
  for (int l = 0; l < a.n_layers; ++l) {
    a.L[l].Wt = ns.sdf.Wt[l], a.L[l].bias = ns.sdf.bias[l], a.L[l].Kpad = ns.sdf.Kpad[l], a.L[l].N = ns.sdf.N[l];
  }
  a.w_last = ns.sdf.w_last, a.b_last = ns.sdf.b_last;
  return HOLD_OK;
}

static int launch_sdf(hold_ctx* ctx, NodeState& ns, int P, const float* xc, const float* embed_w, float* sdf,
                      float* grad, float* feat, const SamplerState* st, cudaStream_t s) {
  if (P <= 0) return HOLD_OK;
  const bool jvp = (grad != nullptr) || (feat != nullptr);
  if (ns.cfg.mlp_mode == HOLD_MLP_TC) return tc_launch_sdf(ctx, ns, P, xc, embed_w, sdf, grad, feat, st, s);
  SimtArgs a;
  memset(&a, 0, sizeof(a));
  fill_sdf_args(ns, a, jvp);
  a.P = P, a.xc = xc, a.embed_w = embed_w, a.sdf = sdf, a.grad = grad, a.feat = feat, a.st = st;
  if (jvp) {
    HOLD_REQUIRE(grad != nullptr && feat != nullptr, "sdf eval with gradient needs both grad and feat buffers");
    int tiles = ceil_div(P, kTileRows / 4);
    k_mlp_simt<MLP_SDF_JVP><<<min(tiles, ctx->sm_count), 256, kSimtSmemBytes, s>>>(a);
  } else {
    int tiles = ceil_div(P, kTileRows);
    k_mlp_simt<MLP_SDF_ONLY><<<min(tiles, ctx->sm_count), 256, kSimtSmemBytes, s>>>(a);
  }
  HOLD_LAUNCH_CHECK(ctx);
  return HOLD_OK;
}

static int launch_rgb(hold_ctx* ctx, NodeState& ns, int P, int pts_per_frame, const float* xc, const float* normal,
                      const float* pe, const float* feat, const float* time_code, float* rgb, cudaStream_t s) {
  if (P <= 0) return HOLD_OK;
  if (ns.cfg.mlp_mode == HOLD_MLP_TC) return tc_launch_rgb(ctx, ns, P, pts_per_frame, xc, normal, pe, feat, time_code, rgb, s);
  SimtArgs a;
  memset(&a, 0, sizeof(a));
  a.n_layers = 4;
  for (int l = 0; l < 4; ++l) {
    a.L[l].Wt = ns.rgb.Wt[l], a.L[l].bias = ns.rgb.bias[l], a.L[l].Kpad = ns.rgb.Kpad[l], a.L[l].N = ns.rgb.N[l];
  }
  a.w_last = ns.rgb.w_last, a.b_last = ns.rgb.b_last;
  a.P = P, a.xc = xc, a.normal = normal, a.pose_embed = pe, a.feat = const_cast<float*>(feat), a.time_code = time_code;
  a.pts_per_frame = pts_per_frame, a.k0 = ns.rgb.K[0], a.rgb = rgb;
  int tiles = ceil_div(P, kTileRows);
  k_mlp_simt<MLP_COLOR><<<min(tiles, ctx->sm_count), 256, kSimtSmemBytes, s>>>(a);
  HOLD_LAUNCH_CHECK(ctx);
  return HOLD_OK;
}

static int launch_inverse_warp(hold_ctx* ctx, NodeState& ns, int B, int pts_per_frame, bool from_z, int nsamp, int zstride,
                               const float* zbuf, const float* cam, const float* dirs, const float* xin,
                               const hold_node_pose* pose, float* xc, int* knn_idx, uint8_t* outlier,
                               const SamplerState* st, cudaStream_t s) {
  if (pts_per_frame <= 0 || B <= 0) return HOLD_OK;
  dim3 grid(ceil_div(pts_per_frame, 128), B);
  const bool hand = ns.cfg.kind == HOLD_KIND_HAND;
  if (hand) {
    HOLD_REQUIRE(pose->posed_verts != nullptr, "hand node needs posed_verts");
    if (!ns.has_rig) { set_error("hand node has no rig (hold_node_set_rig)"); return HOLD_E_STATE; }
  }
  if (hand && from_z && knn_idx == nullptr && outlier == nullptr) {
    // hot path: consecutive samples of a ray per thread, KNN seeded from the previous sample
    const int rays = pts_per_frame / nsamp;
    // walk length per thread: 32 samples when that still fills the GPU (>= 2 waves of 4 blocks per SM), else shorter walks
    int seg_len = kSeg;
    while (seg_len > 4 && (long long)B * rays * ceil_div(nsamp, seg_len) < (long long)ctx->sm_count * 4 * 128 * 2) seg_len >>= 1;
    const int segs = ceil_div(nsamp, seg_len);
    dim3 g2(ceil_div(rays * segs, 128), B);
    k_inverse_warp_hand_rays<<<g2, 128, 0, s>>>(rays, nsamp, seg_len, zstride, zbuf, cam, dirs, pose->tfs, pose->posed_verts, ns.skin_w, ns.knn_perm, xc, st);
    HOLD_LAUNCH_CHECK(ctx);
    return HOLD_OK;
  }
#define IW(H, Z) k_inverse_warp<H, Z><<<grid, 128, 0, s>>>(pts_per_frame, nsamp, zstride, zbuf, cam, dirs, xin, pose->tfs, \
                                                          pose->posed_verts, ns.skin_w, xc, knn_idx, outlier, st, ctx->dev_err)
  if (hand && from_z) IW(true, true);
  else if (hand) IW(true, false);
  else if (from_z) IW(false, true);
  else IW(false, false);
#undef IW
  HOLD_LAUNCH_CHECK(ctx);
  return HOLD_OK;
}

}  // namespace hold

using namespace hold;

// ================================================================================================ C ABI
extern "C" {

int hold_version(void) { return HOLD_B200_VERSION; }
const char* hold_last_error(void) { return g_err; }

int hold_ctx_create(hold_ctx** out, int device) {
  HOLD_REQUIRE(out != nullptr, "out is NULL");
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) {
    set_error("no CUDA device: %s (hold_b200 has no CPU fallback)", cudaGetErrorString(e));
    return HOLD_E_CUDA;
  }
  HOLD_REQUIRE(device >= 0 && device < count, "device %d out of range (%d devices)", device, count);
  HOLD_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  HOLD_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    set_error("device %d is sm_%d%d; hold_b200 is built for sm_100a only", device, prop.major, prop.minor);
    return HOLD_E_CUDA;
  }
  hold_ctx* ctx = new (std::nothrow) hold_ctx();
  if (!ctx) { set_error("out of host memory"); return HOLD_E_NOMEM; }
  ctx->device = device;
  ctx->sm_count = prop.multiProcessorCount;
  HOLD_CUDA(cudaMalloc((void**)&ctx->dev_err, sizeof(int)));
  HOLD_CUDA(cudaMemset(ctx->dev_err, 0, sizeof(int)));
  HOLD_CUDA(cudaFuncSetAttribute(k_mlp_simt<MLP_SDF_ONLY>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSimtSmemBytes));
  HOLD_CUDA(cudaFuncSetAttribute(k_mlp_simt<MLP_SDF_JVP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSimtSmemBytes));
  HOLD_CUDA(cudaFuncSetAttribute(k_mlp_simt<MLP_COLOR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSimtSmemBytes));
  const int samp_smem = 4 * 6 * kMaxZ * (int)sizeof(float);
  HOLD_CUDA(cudaFuncSetAttribute(k_sampler_merge_beta, cudaFuncAttributeMaxDynamicSharedMemorySize, samp_smem));
  HOLD_CUDA(cudaFuncSetAttribute(k_sampler_resample, cudaFuncAttributeMaxDynamicSharedMemorySize, samp_smem));
  const int mano_smem = (2 * kVerts * 3 + kJoints * 3 + kJoints * 9 + 136 + 2 * kJoints * 16 + 16) * (int)sizeof(float);
  (void)mano_smem;
  HOLD_CUDA(cudaFuncSetAttribute(k_bg_mlp<BG_SDF>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kBgSmemBytes));
  HOLD_CUDA(cudaFuncSetAttribute(k_bg_mlp<BG_RGB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kBgSmemBytes));
  int rc = tc_init(ctx);
  if (rc == HOLD_OK) rc = wgrad_init();
  if (rc == HOLD_OK) rc = tc_bg_init();
  if (rc) { delete ctx; return rc; }
  *out = ctx;
  return HOLD_OK;
}

int hold_ctx_destroy(hold_ctx* ctx) {
  if (!ctx) return HOLD_OK;
  cudaSetDevice(ctx->device);
  for (int i = 0; i < 24; ++i)
    if (ctx->ws[i].p) cudaFree(ctx->ws[i].p);
  for (int n = 0; n < HOLD_MAX_NODES; ++n) {
    NodeState& ns = ctx->nodes[n];
    for (int l = 0; l < HOLD_MAX_LAYERS; ++l) {
      if (ns.sdf.Wt[l]) cudaFree(ns.sdf.Wt[l]);
      if (ns.sdf.bias[l]) cudaFree(ns.sdf.bias[l]);
      if (ns.rgb.Wt[l]) cudaFree(ns.rgb.Wt[l]);
      if (ns.rgb.bias[l]) cudaFree(ns.rgb.bias[l]);
    }
    float* ptrs[] = {ns.sdf.w_last, ns.sdf.b_last, ns.rgb.w_last, ns.rgb.b_last, ns.lin_pose_w, ns.lin_pose_b, ns.cano_verts, ns.skin_w};
    for (float* p : ptrs)
      if (p) cudaFree(p);
    if (ns.sstate) cudaFree(ns.sstate);
    if (ns.knn_perm) cudaFree(ns.knn_perm);
    tc_free(ns);
  }
  tc_bg_free(ctx->bg_tc);
  for (int l = 0; l < HOLD_MAX_LAYERS; ++l) {
    if (ctx->bg_sdf.Wt[l]) cudaFree(ctx->bg_sdf.Wt[l]);
    if (ctx->bg_sdf.bias[l]) cudaFree(ctx->bg_sdf.bias[l]);
    if (ctx->bg_rgb.Wt[l]) cudaFree(ctx->bg_rgb.Wt[l]);
    if (ctx->bg_rgb.bias[l]) cudaFree(ctx->bg_rgb.bias[l]);
  }
  {
    float* ptrs[] = {ctx->bg_sdf.w_last, ctx->bg_sdf.b_last, ctx->bg_rgb.w_last, ctx->bg_rgb.b_last};
    for (float* p : ptrs)
      if (p) cudaFree(p);
  }
  if (ctx->dev_err) cudaFree(ctx->dev_err);
  delete ctx;
  return HOLD_OK;
}

int hold_ctx_check(hold_ctx* ctx, void* stream) {
  HOLD_REQUIRE(ctx != nullptr, "ctx is NULL");
  cudaStream_t s = (cudaStream_t)stream;
  int h = 0;
  HOLD_CUDA(cudaMemcpyAsync(&h, ctx->dev_err, sizeof(int), cudaMemcpyDeviceToHost, s));
  HOLD_CUDA(cudaStreamSynchronize(s));
  if (h != 0) HOLD_CUDA(cudaMemsetAsync(ctx->dev_err, 0, sizeof(int), s));
  if (h & 0x100) { set_error("tcgen05 pipeline wait timed out (tag %d): protocol error in k_mlp_tc", (h >> 12) & 0xF); return HOLD_E_STATE; }
  if (h & kErrRayMiss) { set_error("a ray misses the scene bounding sphere (engine/ray_sampler.py:15-18)"); return HOLD_E_RAY_MISSES_SPHERE; }
  if (h & kErrNonFinite) { set_error("non-finite value (singular transform)"); return HOLD_E_NONFINITE; }
  return HOLD_OK;
}

int64_t hold_ctx_launch_count(hold_ctx* ctx) { return ctx ? ctx->launches : -1; }

int hold_node_configure(hold_ctx* ctx, int node, const hold_node_cfg* cfg) {
  HOLD_REQUIRE(ctx != nullptr && cfg != nullptr, "NULL argument");
  HOLD_REQUIRE(node >= 0 && node < HOLD_MAX_NODES, "node %d out of range", node);
  HOLD_REQUIRE(cfg->kind == HOLD_KIND_HAND || cfg->kind == HOLD_KIND_OBJECT, "bad kind %d", cfg->kind);
  HOLD_REQUIRE(cfg->class_id >= 0 && cfg->class_id < 4, "class_id %d out of [0,4)", cfg->class_id);
  HOLD_REQUIRE(cfg->n_samples_eval >= 2 && cfg->max_total_iters >= 1 && cfg->max_total_iters <= 8 &&
                   cfg->n_samples_eval * cfg->max_total_iters <= kMaxZ,
               "sampler buffer: n_samples_eval * max_total_iters must be <= %d", kMaxZ);
  HOLD_REQUIRE(cfg->n_samples >= 1 && cfg->n_samples <= cfg->n_samples_eval * cfg->max_total_iters, "bad n_samples");
  HOLD_REQUIRE(cfg->n_samples + cfg->n_samples_extra + 2 <= 512, "final sample count too large");
  HOLD_REQUIRE(cfg->mlp_mode == HOLD_MLP_FP32 || cfg->mlp_mode == HOLD_MLP_TC, "bad mlp_mode");
  HOLD_CUDA(cudaSetDevice(ctx->device));
  NodeState& ns = ctx->nodes[node];
  ns.cfg = *cfg;
  if (!ns.sstate) HOLD_CUDA(cudaMalloc((void**)&ns.sstate, sizeof(SamplerState)));
  HOLD_CUDA(cudaMemset(ns.sstate, 0, sizeof(SamplerState)));
  ns.configured = true;
  return HOLD_OK;
}

int hold_node_set_weights(hold_ctx* ctx, int node, const hold_mlp_weights* sdf, const hold_mlp_weights* rgb,
                          const float* lin_pose_w, const float* lin_pose_b, void* stream) {
  int rc = check_node(ctx, node, false);
  if (rc) return rc;
  HOLD_REQUIRE(sdf != nullptr && rgb != nullptr, "NULL weights");
  NodeState& ns = ctx->nodes[node];
  cudaStream_t s = (cudaStream_t)stream;
  const bool hand = ns.cfg.kind == HOLD_KIND_HAND;
  // ---- SDF net: dims [39(+45)] ->256 x3 -> 217 (+39) ->256 x4 -> 257 (networks/shape_net.py:13-49)
  HOLD_REQUIRE(sdf->n_layers == 9, "SDF net must have 9 layers, got %d", sdf->n_layers);
  HOLD_REQUIRE(sdf->in_dim[0] == (hand ? kEmbed + 45 : kEmbed), "SDF lin0 in_dim %d unexpected for this node kind", sdf->in_dim[0]);
  for (int l = 0; l < 9; ++l) {
    int eo = (l == 3) ? kHidden - kEmbed : (l == 8 ? kFeat + 1 : kHidden);
    int ei = (l == 0) ? sdf->in_dim[0] : kHidden;
    HOLD_REQUIRE(sdf->out_dim[l] == eo && sdf->in_dim[l] == ei, "SDF lin%d is %dx%d, expected %dx%d", l, sdf->out_dim[l], sdf->in_dim[l], eo, ei);
    HOLD_REQUIRE(sdf->weight_v[l] && sdf->bias[l], "SDF lin%d has NULL tensors", l);
  }
  for (int l = 0; l < 9; ++l) {
    int K = (l == 0) ? kEmbed : kHidden;
    int Kpad = round_up(K, kKC);
    int N = (l == 3) ? kHidden - kEmbed : kHidden;
    int row_off = (l == 8) ? 1 : 0;  // lin8 row 0 is the sdf head, rows 1..256 the feature vector
    ns.sdf.K[l] = K, ns.sdf.N[l] = N, ns.sdf.Kpad[l] = Kpad, ns.sdf.Npad[l] = 256;
    rc = dev_alloc(&ns.sdf.Wt[l], (size_t)Kpad * 256);
    if (rc) return rc;
    rc = dev_alloc(&ns.sdf.bias[l], 256);
    if (rc) return rc;
    float scale = (l == 4) ? (float)(1.0 / sqrt(2.0)) : 1.0f;  // skip_in: cat([x, input]) / sqrt(2)
    k_pack_layer<<<256, 128, 0, s>>>(sdf->weight_v[l], sdf->weight_g[l], sdf->bias[l], sdf->in_dim[l], row_off, 0, K, N,
                                     Kpad, scale, ns.sdf.Wt[l], ns.sdf.bias[l]);
    HOLD_LAUNCH_CHECK(ctx);
  }
  ns.sdf.n_layers = 9;
  rc = dev_alloc(&ns.sdf.w_last, 256);
  if (rc) return rc;
  rc = dev_alloc(&ns.sdf.b_last, 4);
  if (rc) return rc;
  k_pack_rows<<<1, 128, 0, s>>>(sdf->weight_v[8], sdf->weight_g[8], sdf->bias[8], 256, 0, 1, ns.sdf.w_last, ns.sdf.b_last);
  HOLD_LAUNCH_CHECK(ctx);
  // ---- colour net: [270|302] -> 256 x4 -> 3 (networks/texture_net.py:13-44)
  HOLD_REQUIRE(rgb->n_layers == 5, "colour net must have 5 layers, got %d", rgb->n_layers);
  const int k0 = hand ? 270 : 302;
  HOLD_REQUIRE(rgb->in_dim[0] == k0, "colour lin0 in_dim %d, expected %d", rgb->in_dim[0], k0);
  for (int l = 0; l < 5; ++l) {
    int eo = (l == 4) ? 3 : 256, ei = (l == 0) ? k0 : 256;
    HOLD_REQUIRE(rgb->out_dim[l] == eo && rgb->in_dim[l] == ei, "colour lin%d is %dx%d, expected %dx%d", l, rgb->out_dim[l], rgb->in_dim[l], eo, ei);
    HOLD_REQUIRE(rgb->weight_v[l] && rgb->bias[l], "colour lin%d has NULL tensors", l);
  }
  for (int l = 0; l < 4; ++l) {
    int K = (l == 0) ? k0 : 256, Kpad = round_up(K, kKC);
    ns.rgb.K[l] = K, ns.rgb.N[l] = 256, ns.rgb.Kpad[l] = Kpad, ns.rgb.Npad[l] = 256;
    rc = dev_alloc(&ns.rgb.Wt[l], (size_t)Kpad * 256);
    if (rc) return rc;
    rc = dev_alloc(&ns.rgb.bias[l], 256);
    if (rc) return rc;
    k_pack_layer<<<256, 128, 0, s>>>(rgb->weight_v[l], rgb->weight_g[l], rgb->bias[l], rgb->in_dim[l], 0, 0, K, 256, Kpad,
                                     1.0f, ns.rgb.Wt[l], ns.rgb.bias[l]);
    HOLD_LAUNCH_CHECK(ctx);
  }
  ns.rgb.n_layers = 5;
  rc = dev_alloc(&ns.rgb.w_last, 3 * 256);
  if (rc) return rc;
  rc = dev_alloc(&ns.rgb.b_last, 4);
  if (rc) return rc;
  k_pack_rows<<<3, 128, 0, s>>>(rgb->weight_v[4], rgb->weight_g[4], rgb->bias[4], 256, 0, 3, ns.rgb.w_last, ns.rgb.b_last);
  HOLD_LAUNCH_CHECK(ctx);
  if (hand) {
    HOLD_REQUIRE(lin_pose_w && lin_pose_b, "hand node needs lin_pose weights");
    rc = dev_alloc(&ns.lin_pose_w, 8 * 45);
    if (rc) return rc;
    rc = dev_alloc(&ns.lin_pose_b, 8);
    if (rc) return rc;
    HOLD_CUDA(cudaMemcpyAsync(ns.lin_pose_w, lin_pose_w, 8 * 45 * sizeof(float), cudaMemcpyDeviceToDevice, s));
    HOLD_CUDA(cudaMemcpyAsync(ns.lin_pose_b, lin_pose_b, 8 * sizeof(float), cudaMemcpyDeviceToDevice, s));
  }
  rc = tc_pack(ctx, ns, sdf, rgb, s);
  if (rc) return rc;
  ns.has_weights = true;
  return HOLD_OK;
}

int hold_node_set_rig(hold_ctx* ctx, int node, const float* cano_verts, const float* skin_weights, void* stream) {
  int rc = check_node(ctx, node, false);
  if (rc) return rc;
  HOLD_REQUIRE(cano_verts && skin_weights, "NULL rig tensors");
  NodeState& ns = ctx->nodes[node];
  HOLD_REQUIRE(ns.cfg.kind == HOLD_KIND_HAND, "only hand nodes have a rig");
  cudaStream_t s = (cudaStream_t)stream;
  rc = dev_alloc(&ns.cano_verts, kVerts * 3);
  if (rc) return rc;
  rc = dev_alloc(&ns.skin_w, kVerts * kJoints);
  if (rc) return rc;
  HOLD_CUDA(cudaMemcpyAsync(ns.cano_verts, cano_verts, kVerts * 3 * sizeof(float), cudaMemcpyDeviceToDevice, s));
  HOLD_CUDA(cudaMemcpyAsync(ns.skin_w, skin_weights, kVerts * kJoints * sizeof(float), cudaMemcpyDeviceToDevice, s));
  {  // vertex groups of the cluster-pruned KNN (knn_phases.h): ordered once on the canonical hand, on the host
    static_assert(knnc::kNV == kVerts && knnc::kK == kKnn, "knn_phases.h constants");
    float* hv = (float*)malloc(sizeof(float) * kVerts * (3 + kJoints));
    HOLD_REQUIRE(hv != nullptr, "out of host memory");
    cudaError_t e = cudaMemcpyAsync(hv, ns.cano_verts, kVerts * 3 * sizeof(float), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(hv + kVerts * 3, ns.skin_w, kVerts * kJoints * sizeof(float), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    unsigned short perm[knnc::kNCl * knnc::kClSize];
    if (e == cudaSuccess) {
      knnc::cluster_order(hv, hv + kVerts * 3, kJoints, perm);
      if (!ns.knn_perm) e = cudaMalloc((void**)&ns.knn_perm, sizeof(perm));
      if (e == cudaSuccess) e = cudaMemcpyAsync(ns.knn_perm, perm, sizeof(perm), cudaMemcpyHostToDevice, s);
      if (e == cudaSuccess) e = cudaStreamSynchronize(s);   // `perm` is a stack buffer
    }
    free(hv);
    if (e != cudaSuccess) { set_error("hold_node_set_rig: %s", cudaGetErrorString(e)); return HOLD_E_CUDA; }
  }
  ns.has_rig = true;
  return HOLD_OK;
}

int hold_mano_lbs(hold_ctx* ctx, const hold_mano_model* m, int B, const float* betas, const float* full_pose,
                  const float* transl, const float* scene_scale, const float* tfs_c_inv, float* verts, float* jnts,
                  float* tfs, float* v_posed, void* stream) {
  HOLD_REQUIRE(ctx && m, "NULL argument");
  HOLD_CUDA(cudaSetDevice(ctx->device));
  HOLD_REQUIRE(B >= 0, "negative batch");
  if (B == 0) return HOLD_OK;
  HOLD_REQUIRE(betas && full_pose && transl && scene_scale && verts && jnts && tfs && v_posed, "NULL tensor");
  HOLD_REQUIRE(m->parents_host && m->tip_ids_host, "NULL host arrays in mano model");
  ManoDev d;
  d.v_template = m->v_template, d.shapedirs = m->shapedirs, d.posedirs = m->posedirs, d.J_regressor = m->J_regressor;
  d.lbs_weights = m->lbs_weights, d.hands_mean = m->hands_mean;
  for (int i = 0; i < kJoints; ++i) {
    d.parents[i] = (i == 0) ? 0 : m->parents_host[i];
    HOLD_REQUIRE(i == 0 || (d.parents[i] >= 0 && d.parents[i] < i), "parents must be topologically ordered");
  }
  for (int i = 0; i < 5; ++i) {
    d.tips[i] = m->tip_ids_host[i];
    HOLD_REQUIRE(d.tips[i] >= 0 && d.tips[i] < kVerts, "tip id out of range");
  }
  constexpr int smem = (2 * kVerts * 3 + kJoints * 3 + kJoints * 9 + 136 + 2 * kJoints * 16 + 16) * (int)sizeof(float);
  static_assert(smem <= 48 * 1024, "k_mano_lbs fits the default dynamic shared memory limit (no per-device attribute needed)");
  k_mano_lbs<<<B, 256, smem, (cudaStream_t)stream>>>(d, betas, full_pose, transl, scene_scale, tfs_c_inv, verts, jnts, tfs, v_posed);
  HOLD_LAUNCH_CHECK(ctx);
  return HOLD_OK;
}

int hold_mano_lbs_bwd(hold_ctx* ctx, const hold_mano_model* m, int B, const float* betas, const float* full_pose,
                      const float* transl, const float* scene_scale, const float* tfs_c_inv, const float* g_verts,
                      const float* g_jnts, const float* g_tfs, float* g_betas, float* g_pose, float* g_transl, float* g_scale,
                      void* stream) {
  HOLD_REQUIRE(ctx && m, "NULL argument");
  HOLD_CUDA(cudaSetDevice(ctx->device));
  HOLD_REQUIRE(B >= 0, "negative batch");
  if (B == 0) return HOLD_OK;
  HOLD_REQUIRE(betas && full_pose && transl && scene_scale && g_betas && g_pose && g_transl && g_scale, "NULL tensor");
  HOLD_REQUIRE(m->parents_host && m->tip_ids_host, "NULL host arrays in mano model");
  posebwd::ManoPtrs d;
  d.v_template = m->v_template, d.shapedirs = m->shapedirs, d.posedirs = m->posedirs, d.J_regressor = m->J_regressor;
  d.lbs_weights = m->lbs_weights, d.hands_mean = m->hands_mean;
  for (int i = 0; i < kJoints; ++i) {
    d.parents[i] = (i == 0) ? 0 : m->parents_host[i];
    HOLD_REQUIRE(i == 0 || (d.parents[i] >= 0 && d.parents[i] < i), "parents must be topologically ordered");
  }
  for (int i = 0; i < 5; ++i) {
    d.tips[i] = m->tip_ids_host[i];
    HOLD_REQUIRE(d.tips[i] >= 0 && d.tips[i] < kVerts, "tip id out of range");
  }
  const int nt = 256, smem = posebwd::mano_scratch_floats(nt) * (int)sizeof(float);
  HOLD_REQUIRE(smem <= 48 * 1024, "k_mano_lbs_bwd scratch exceeds the default dynamic shared memory limit");
  k_mano_lbs_bwd<<<B, nt, smem, (cudaStream_t)stream>>>(d, betas, full_pose, transl, scene_scale, tfs_c_inv, g_verts, g_jnts, g_tfs,
                                                        g_betas, g_pose, g_transl, g_scale);
  HOLD_LAUNCH_CHECK(ctx);
  return HOLD_OK;
}

int hold_object_tf_bwd(hold_ctx* ctx, int B, const float* rot, const float* trans, const float* scene_scale, float obj_scale,
                       const float* denorm_mat, const float* pts_cano, int Nv, const float* g_verts, const float* g_tfs,
                       float* g_rot, float* g_trans, float* g_scene_scale, float* g_obj_scale, void* stream) {
  HOLD_REQUIRE(ctx && rot && trans && scene_scale && denorm_mat && g_rot && g_trans && g_scene_scale && g_obj_scale, "NULL argument");
  HOLD_CUDA(cudaSetDevice(ctx->device));
  if (B <= 0) return HOLD_OK;
  HOLD_REQUIRE(g_verts == nullptr || (pts_cano != nullptr && Nv > 0), "g_verts given without canonical points");
  const int nt = 256, smem = posebwd::obj_scratch_floats(nt) * (int)sizeof(float);
  k_object_tf_bwd<<<B, nt, smem, (cudaStream_t)stream>>>(Nv, rot, trans, scene_scale, obj_scale, denorm_mat, pts_cano, g_verts, g_tfs,
                                                         g_rot, g_trans, g_scene_scale, g_obj_scale);
  HOLD_LAUNCH_CHECK(ctx);
  return HOLD_OK;
}

int hold_object_tf(hold_ctx* ctx, int B, const float* rot, const float* trans, const float* scene_scale, float obj_scale,
                   const float* denorm_mat, const float* pts_cano, int Nv, float* tfs, float* verts, void* stream) {
  HOLD_REQUIRE(ctx && rot && trans && scene_scale && denorm_mat && tfs, "NULL argument");
  HOLD_CUDA(cudaSetDevice(ctx->device));
  if (B <= 0) return HOLD_OK;
  HOLD_REQUIRE(verts == nullptr || (pts_cano != nullptr && Nv > 0), "verts requested without canonical points");
  dim3 grid(verts ? max(1, min(ceil_div(Nv, 128), 64)) : 1, B);
  k_object_tf<<<grid, 128, 0, (cudaStream_t)stream>>>(B, Nv, rot, trans, scene_scale, obj_scale, denorm_mat, pts_cano, tfs, verts);
  HOLD_LAUNCH_CHECK(ctx);
  return HOLD_OK;
}

int hold_camera_rays(hold_ctx* ctx, int B, int P, const float* uv, const float* pose, const float* intrinsics,
                     float* ray_dirs, float* cam_loc, void* stream) {
  HOLD_REQUIRE(ctx && uv && pose && intrinsics && ray_dirs && cam_loc, "NULL argument");
  HOLD_CUDA(cudaSetDevice(ctx->device));
  if (B * P <= 0) return HOLD_OK;
  k_camera_rays<<<ceil_div(B * P, 256), 256, 0, (cudaStream_t)stream>>>(B, P, uv, pose, intrinsics, ray_dirs, cam_loc);
  HOLD_LAUNCH_CHECK(ctx);
  return HOLD_OK;
}

int hold_sample(hold_ctx* ctx, int node, int R, int B, const float* cam_loc, const float* ray_dirs,
                const hold_node_pose* pose, const hold_sampler_rand* rnd, float* z_vals, int32_t* iters, void* stream) {
  int rc = check_node(ctx, node, true);
  if (rc) return rc;
  HOLD_REQUIRE(R >= 0 && B >= 1, "bad R/B");
  if (R == 0) return HOLD_OK;
  HOLD_REQUIRE(R % B == 0, "R (%d) must be B (%d) frames x rays, frame-major", R, B);
  HOLD_REQUIRE(cam_loc && ray_dirs && pose && z_vals, "NULL argument");
  HOLD_REQUIRE(pose->tfs && pose->beta_param, "pose needs tfs and beta_param");
  NodeState& ns = ctx->nodes[node];
  const hold_node_cfg& c = ns.cfg;
  cudaStream_t s = (cudaStream_t)stream;
  const int Ne = c.n_samples_eval;
  WS(WS_Z, float, (size_t)R * kMaxZ, zb);
  WS(WS_SDF, float, (size_t)R * kMaxZ, sb);
  WS(WS_ZNEW, float, (size_t)R * Ne, znew);
  WS(WS_SDFNEW, float, (size_t)R * Ne, sdfnew);
  WS(WS_BETA, float, R, betab);
  WS(WS_FAR, float, R, farb);
  WS(WS_XC, float, (size_t)R * Ne * 3, xc);
  SamplerArgs a;
  memset(&a, 0, sizeof(a));
  a.R = R, a.rays_per_frame = R / B;
  a.n_eval = Ne, a.n_samples = c.n_samples, a.n_extra = c.n_samples_extra, a.beta_iters = c.beta_iters, a.max_iters = c.max_total_iters;
  a.eps = c.eps, a.add_tiny = c.add_tiny, a.near = c.near, a.r_sphere = c.bounding_sphere, a.beta_min = c.beta_min;
  a.cam = cam_loc, a.dirs = ray_dirs, a.beta_param = pose->beta_param;
  a.z = zb, a.sdf = sb, a.znew = znew, a.sdfnew = sdfnew, a.beta = betab, a.far = farb, a.st = ns.sstate, a.err = ctx->dev_err;
  if (rnd) { a.jitter = rnd->jitter, a.u_rand = rnd->u, a.extra_idx = rnd->extra_idx; }
  a.z_out = z_vals, a.iters_out = iters;
  const int wpb = 4;
  k_sampler_init<<<ceil_div(R, wpb), wpb * 32, 0, s>>>(a);
  HOLD_LAUNCH_CHECK(ctx);
  for (int it = 0; it < c.max_total_iters; ++it) {
    if (it > 0) {
      k_round_gate<<<1, 1, 0, s>>>(ns.sstate, it, pose->beta_param, c.beta_min, c.max_total_iters);
      HOLD_LAUNCH_CHECK(ctx);
    }
    rc = launch_inverse_warp(ctx, ns, B, (R / B) * Ne, true, Ne, Ne, znew, cam_loc, ray_dirs, nullptr, pose, xc, nullptr,
                             nullptr, ns.sstate, s);
    if (rc) return rc;
    rc = launch_sdf(ctx, ns, R * Ne, xc, pose->embed_w, sdfnew, nullptr, nullptr, ns.sstate, s);
    if (rc) return rc;
    const int cap = sampler_cap(it, Ne, c.n_samples + c.n_samples_extra + 2);
    const int samp_smem = wpb * 6 * cap * (int)sizeof(float);
    k_sampler_merge_beta<<<ceil_div(R, wpb), wpb * 32, samp_smem, s>>>(a, it, cap);
    HOLD_LAUNCH_CHECK(ctx);
    k_sampler_resample<<<ceil_div(R, wpb), wpb * 32, samp_smem, s>>>(a, it, cap);
    HOLD_LAUNCH_CHECK(ctx);
  }
  return HOLD_OK;
}

/* One iteration of the while loop of ErrorBoundSampler.get_z_vals (engine/ray_sampler.py:160-311) on caller-supplied state:
 * the sorted (z, sdf) of the previous rounds, this round's new samples and their sdf, beta per ray.  Runs exactly the kernels
 * hold_sample runs for round `it` (merge + d* + beta line search, then PDF -> inverse CDF), so that a round can be compared
 * with the reference in isolation (teacher forcing): upstream last-bit differences do not propagate into it. */
int hold_sampler_round(hold_ctx* ctx, int node, int R, int it, const float* z_old, const float* sdf_old, const float* z_new,
                       const float* sdf_new, const float* beta_in, const float* far, const float* beta_param,
                       float* z_merged, float* sdf_merged, float* beta_out, float* samples_out, int32_t* upsample_out,
                       void* stream) {
  int rc = check_node(ctx, node, false);
  if (rc) return rc;
  NodeState& ns = ctx->nodes[node];
  const hold_node_cfg& c = ns.cfg;
  HOLD_REQUIRE(R >= 0 && it >= 0 && it < c.max_total_iters, "bad R / round index");
  if (R == 0) return HOLD_OK;
  HOLD_REQUIRE(z_new && sdf_new && beta_in && far && beta_param && beta_out && samples_out, "NULL argument");
  HOLD_REQUIRE(it == 0 || (z_old && sdf_old), "round %d needs the previous rounds' (z, sdf)", it);
  HOLD_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t s = (cudaStream_t)stream;
  const int Ne = c.n_samples_eval, n_old = it * Ne, n = n_old + Ne;
  WS(WS_Z, float, (size_t)R * kMaxZ, zb);
  WS(WS_SDF, float, (size_t)R * kMaxZ, sb);
  WS(WS_ZNEW, float, (size_t)R * Ne, znew);
  WS(WS_SDFNEW, float, (size_t)R * Ne, sdfnew);
  WS(WS_BETA, float, R, betab);
  WS(WS_FAR, float, R, farb);
  WS(WS_ZTMP, float, (size_t)R * 512, zfin);
  if (n_old > 0) {
    HOLD_CUDA(cudaMemcpy2DAsync(zb, kMaxZ * sizeof(float), z_old, n_old * sizeof(float), n_old * sizeof(float), R, cudaMemcpyDeviceToDevice, s));
    HOLD_CUDA(cudaMemcpy2DAsync(sb, kMaxZ * sizeof(float), sdf_old, n_old * sizeof(float), n_old * sizeof(float), R, cudaMemcpyDeviceToDevice, s));
  }
  HOLD_CUDA(cudaMemcpyAsync(znew, z_new, (size_t)R * Ne * sizeof(float), cudaMemcpyDeviceToDevice, s));
  HOLD_CUDA(cudaMemcpyAsync(sdfnew, sdf_new, (size_t)R * Ne * sizeof(float), cudaMemcpyDeviceToDevice, s));
  HOLD_CUDA(cudaMemcpyAsync(betab, beta_in, (size_t)R * sizeof(float), cudaMemcpyDeviceToDevice, s));
  HOLD_CUDA(cudaMemcpyAsync(farb, far, (size_t)R * sizeof(float), cudaMemcpyDeviceToDevice, s));
  HOLD_CUDA(cudaMemsetAsync(ns.sstate, 0, sizeof(SamplerState), s));
  SamplerArgs a;
  memset(&a, 0, sizeof(a));
  a.R = R, a.rays_per_frame = R;
  a.n_eval = Ne, a.n_samples = c.n_samples, a.n_extra = c.n_samples_extra, a.beta_iters = c.beta_iters, a.max_iters = c.max_total_iters;
  a.eps = c.eps, a.add_tiny = c.add_tiny, a.near = c.near, a.r_sphere = c.bounding_sphere, a.beta_min = c.beta_min;
  a.beta_param = beta_param;
  a.z = zb, a.sdf = sb, a.znew = znew, a.sdfnew = sdfnew, a.beta = betab, a.far = farb, a.st = ns.sstate, a.err = ctx->dev_err;
  a.z_out = zfin, a.iters_out = nullptr;
  const int wpb = 4;
  const int cap = sampler_cap(it, Ne, c.n_samples + c.n_samples_extra + 2);
  const int samp_smem = wpb * 6 * cap * (int)sizeof(float);
  k_sampler_merge_beta<<<ceil_div(R, wpb), wpb * 32, samp_smem, s>>>(a, it, cap);
  HOLD_LAUNCH_CHECK(ctx);
  if (z_merged) HOLD_CUDA(cudaMemcpy2DAsync(z_merged, n * sizeof(float), zb, kMaxZ * sizeof(float), n * sizeof(float), R, cudaMemcpyDeviceToDevice, s));
  if (sdf_merged) HOLD_CUDA(cudaMemcpy2DAsync(sdf_merged, n * sizeof(float), sb, kMaxZ * sizeof(float), n * sizeof(float), R, cudaMemcpyDeviceToDevice, s));
  HOLD_CUDA(cudaMemcpyAsync(beta_out, betab, (size_t)R * sizeof(float), cudaMemcpyDeviceToDevice, s));
  k_sampler_resample<<<ceil_div(R, wpb), wpb * 32, samp_smem, s>>>(a, it, cap);
  HOLD_LAUNCH_CHECK(ctx);
  // upsample decision of this round (ray_sampler.py:244-246), read back for the caller: it sizes samples_out
  unsigned int bits = 0;
  float b0 = 0.f;
  HOLD_CUDA(cudaMemcpyAsync(&bits, &ns.sstate->beta_max_bits[it], sizeof(bits), cudaMemcpyDeviceToHost, s));
  HOLD_CUDA(cudaMemcpyAsync(&b0, beta_param, sizeof(float), cudaMemcpyDeviceToHost, s));
  HOLD_CUDA(cudaStreamSynchronize(s));
  float bm;
  memcpy(&bm, &bits, sizeof(bm));
  const bool upsample = (bm > fabsf(b0) + c.beta_min) && (it + 1 < c.max_total_iters);
  if (upsample_out) *upsample_out = upsample ? 1 : 0;
  if (upsample) {
    HOLD_CUDA(cudaMemcpyAsync(samples_out, znew, (size_t)R * Ne * sizeof(float), cudaMemcpyDeviceToDevice, s));
  } else {
    const int S = c.n_samples + c.n_samples_extra + 2;
    HOLD_CUDA(cudaMemcpyAsync(samples_out, zfin, (size_t)R * S * sizeof(float), cudaMemcpyDeviceToDevice, s));
  }
  return HOLD_OK;
}

int hold_shade(hold_ctx* ctx, int node, int R, int B, int S, const float* cam_loc, const float* ray_dirs,
               const hold_node_pose* pose, const hold_factors* out, void* stream) {
  int rc = check_node(ctx, node, true);
  if (rc) return rc;
  HOLD_REQUIRE(R >= 0 && B >= 1 && S >= 1, "bad R/B/S");
  if (R == 0) return HOLD_OK;
  HOLD_REQUIRE(R % B == 0, "R (%d) must be B (%d) frames x rays, frame-major", R, B);
  HOLD_REQUIRE(cam_loc && ray_dirs && pose && out, "NULL argument");
  HOLD_REQUIRE(out->z_vals && out->color && out->normal && out->density, "factors need z_vals, color, normal, density");
  HOLD_REQUIRE(pose->tfs && pose->beta_param, "pose needs tfs and beta_param");
  NodeState& ns = ctx->nodes[node];
  const bool hand = ns.cfg.kind == HOLD_KIND_HAND;
  if (!hand) HOLD_REQUIRE(pose->time_code != nullptr, "object node needs time_code");
  cudaStream_t s = (cudaStream_t)stream;
  const int rpf = R / B;
  const int max_pts = 1 << 20;
  const int rays_per_chunk = max(1, min(rpf, max_pts / S));
  const size_t cp = (size_t)rays_per_chunk * S;
  // canonical points of the WHOLE call in one launch (full grid, one vertex-group setup per block instead of one per 1 Mi-point
  // chunk: the per-chunk launches of round 1 ran at 0.57 waves); the MLP stages below are chunked for their 1 GB feature buffer
  float* xc_all = out->canonical_pts;
  if (xc_all == nullptr) {
    WS(WS_XC, float, (size_t)R * S * 3, xc_ws);
    xc_all = xc_ws;
  }
  WS(WS_SSDF, float, cp, sdf_ws);
  WS(WS_GRAD, float, cp * 3, grad_ws);
  WS(WS_FEAT, float, cp * kFeat, feat_ws);
  float* pe = nullptr;
  if (hand && pose->pose_cond != nullptr) {
    WS(WS_PE, float, (size_t)B * 8, pe_ws);
    pe = pe_ws;
    k_pose_embed<<<ceil_div(B * 8, 64), 64, 0, s>>>(B, pose->pose_cond, ns.lin_pose_w, ns.lin_pose_b, pe);
    HOLD_LAUNCH_CHECK(ctx);
  } else if (hand) {
    // RenderingNet with a 45-dim pose of zeros still applies lin_pose: embed = bias (texture_net.py:80-82)
    HOLD_REQUIRE(false, "hand node needs pose_cond (pass zeros for the first 20 training epochs)");
  }
  rc = launch_inverse_warp(ctx, ns, B, rpf * S, true, S, S, out->z_vals, cam_loc, ray_dirs, nullptr, pose, xc_all, nullptr, nullptr, nullptr, s);
  if (rc) return rc;
  for (int b = 0; b < B; ++b) {
    hold_node_pose pb = *pose;
    pb.tfs = pose->tfs + (size_t)b * (hand ? kJoints * 16 : 16);
    if (hand) pb.posed_verts = pose->posed_verts + (size_t)b * kVerts * 3;
    for (int r0 = 0; r0 < rpf; r0 += rays_per_chunk) {
      const int rc_n = min(rays_per_chunk, rpf - r0);
      const size_t ray0 = (size_t)b * rpf + r0;
      const int P = rc_n * S;
      float* xc = xc_all + ray0 * S * 3;
      float* sdf = out->sdf ? out->sdf + ray0 * S : sdf_ws;
      rc = launch_sdf(ctx, ns, P, xc, pose->embed_w, sdf, grad_ws, feat_ws, nullptr, s);
      if (rc) return rc;
      dim3 grid(ceil_div(P, 128), 1);
      if (hand)
        k_normals_density<true><<<grid, 128, 0, s>>>(P, xc, grad_ws, sdf, pb.tfs, ns.cano_verts, ns.skin_w, pose->beta_param,
                                                    ns.cfg.beta_min, out->normal + ray0 * S * 3, out->density + ray0 * S);
      else
        k_normals_density<false><<<grid, 128, 0, s>>>(P, xc, grad_ws, sdf, pb.tfs, nullptr, nullptr, pose->beta_param,
                                                     ns.cfg.beta_min, out->normal + ray0 * S * 3, out->density + ray0 * S);
      HOLD_LAUNCH_CHECK(ctx);
      rc = launch_rgb(ctx, ns, P, P, xc, out->normal + ray0 * S * 3, pe ? pe + b * 8 : nullptr, feat_ws,
                      hand ? nullptr : pose->time_code + b * 32, out->color + ray0 * S * 3, s);
      if (rc) return rc;
    }
  }
  return HOLD_OK;
}

int hold_composite(hold_ctx* ctx, int n, int R, int S, const hold_factors* factors, const int32_t* class_ids_host,
                   const hold_render_out* comp, const hold_render_out* per_node, void* stream) {
  HOLD_REQUIRE(ctx && factors && class_ids_host, "NULL argument");
  HOLD_CUDA(cudaSetDevice(ctx->device));
  HOLD_REQUIRE(n >= 1 && n <= HOLD_MAX_NODES, "n = %d out of [1,%d]", n, HOLD_MAX_NODES);
  HOLD_REQUIRE(R >= 0 && S >= 2, "bad R/S");
  if (R == 0) return HOLD_OK;
  cudaStream_t s = (cudaStream_t)stream;
  CompositeArgs a;
  memset(&a, 0, sizeof(a));
  a.R = R, a.S = S;
  for (int k = 0; k < n; ++k) {
    HOLD_REQUIRE(factors[k].color && factors[k].normal && factors[k].density && factors[k].z_vals, "factors[%d] incomplete", k);
    HOLD_REQUIRE(class_ids_host[k] >= 0 && class_ids_host[k] < 4, "class id out of range");
  }
  if (comp != nullptr) {
    a.n = n;
    for (int k = 0; k < n; ++k) {
      a.color[k] = factors[k].color, a.normal[k] = factors[k].normal, a.density[k] = factors[k].density, a.z[k] = factors[k].z_vals;
      a.class_id[k] = class_ids_host[k];
    }
    a.out = *comp, a.drop_head = n - 1, a.drop_tail = n, a.single_zmax_last = 0;
    k_composite<<<ceil_div(R, 128), 128, 0, s>>>(a);
    HOLD_LAUNCH_CHECK(ctx);
  }
  if (per_node != nullptr) {
    for (int k = 0; k < n; ++k) {
      CompositeArgs b;
      memset(&b, 0, sizeof(b));
      b.R = R, b.S = S, b.n = 1;
      b.color[0] = factors[k].color, b.normal[0] = factors[k].normal, b.density[0] = factors[k].density, b.z[0] = factors[k].z_vals;
      b.class_id[0] = class_ids_host[k];
      b.out = per_node[k], b.drop_head = 0, b.drop_tail = 0, b.single_zmax_last = 1;
      k_composite<<<ceil_div(R, 128), 128, 0, s>>>(b);
      HOLD_LAUNCH_CHECK(ctx);
    }
  }
  return HOLD_OK;
}

int hold_composite_bwd(hold_ctx* ctx, int n, int R, int S, const hold_factors* factors, const int32_t* class_ids_host,
                       const hold_render_out* g_comp, const hold_render_out* g_per_node, const hold_factors* d_factors, void* stream) {
  HOLD_REQUIRE(ctx && factors && class_ids_host && d_factors, "NULL argument");
  HOLD_REQUIRE(n >= 1 && n <= HOLD_MAX_NODES, "n = %d out of [1,%d]", n, HOLD_MAX_NODES);
  HOLD_REQUIRE(R >= 0 && S >= 2, "bad R/S");
  HOLD_REQUIRE(g_comp != nullptr || g_per_node != nullptr, "no upstream gradient given");
  if (R == 0) return HOLD_OK;
  HOLD_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t s = (cudaStream_t)stream;
  for (int k = 0; k < n; ++k) {
    HOLD_REQUIRE(factors[k].color && factors[k].normal && factors[k].density && factors[k].z_vals, "factors[%d] incomplete", k);
    HOLD_REQUIRE(d_factors[k].color && d_factors[k].normal && d_factors[k].density, "d_factors[%d] needs color, normal, density", k);
    HOLD_REQUIRE(class_ids_host[k] >= 0 && class_ids_host[k] < 4, "class id out of range");
  }
  bool written = false;
  if (g_comp != nullptr) {
    CompositeBwdArgs a;
    memset(&a, 0, sizeof(a));
    a.n = n, a.R = R, a.S = S;
    for (int k = 0; k < n; ++k) {
      a.color[k] = factors[k].color, a.normal[k] = factors[k].normal, a.density[k] = factors[k].density, a.z[k] = factors[k].z_vals;
      a.class_id[k] = class_ids_host[k];
      a.d_color[k] = d_factors[k].color, a.d_normal[k] = d_factors[k].normal, a.d_density[k] = d_factors[k].density;
    }
    a.g = *g_comp, a.drop_head = n - 1, a.drop_tail = n, a.single_zmax_last = 0, a.accumulate = 0;
    k_composite_bwd<<<ceil_div(R, 128), 128, 0, s>>>(a);
    HOLD_LAUNCH_CHECK(ctx);
    written = true;
  }
  if (g_per_node != nullptr) {
    for (int k = 0; k < n; ++k) {
      CompositeBwdArgs b;
      memset(&b, 0, sizeof(b));
      b.n = 1, b.R = R, b.S = S;
      b.color[0] = factors[k].color, b.normal[0] = factors[k].normal, b.density[0] = factors[k].density, b.z[0] = factors[k].z_vals;
      b.class_id[0] = class_ids_host[k];
      b.d_color[0] = d_factors[k].color, b.d_normal[0] = d_factors[k].normal, b.d_density[0] = d_factors[k].density;
      b.g = g_per_node[k], b.drop_head = 0, b.drop_tail = 0, b.single_zmax_last = 1, b.accumulate = written ? 1 : 0;
      k_composite_bwd<<<ceil_div(R, 128), 128, 0, s>>>(b);
      HOLD_LAUNCH_CHECK(ctx);
    }
  }
  return HOLD_OK;
}

int hold_render_fg(hold_ctx* ctx, int n, const int32_t* node_ids_host, int R, int B, const float* cam_loc,
                   const float* ray_dirs, const hold_node_pose* poses, const hold_factors* factors,
                   const hold_render_out* comp, const hold_render_out* per_node, int32_t* iters, void* stream) {
  HOLD_REQUIRE(ctx && node_ids_host && poses && factors, "NULL argument");
  HOLD_REQUIRE(n >= 1 && n <= HOLD_MAX_NODES, "n = %d out of [1,%d]", n, HOLD_MAX_NODES);
  int32_t cls[HOLD_MAX_NODES];
  int S = -1;
  for (int k = 0; k < n; ++k) {
    int node = node_ids_host[k];
    int rc = check_node(ctx, node, true);
    if (rc) return rc;
    const hold_node_cfg& c = ctx->nodes[node].cfg;
    int Sk = c.n_samples + c.n_samples_extra + 2;
    HOLD_REQUIRE(S < 0 || S == Sk, "all nodes must produce the same number of samples per ray");
    S = Sk;
    cls[k] = c.class_id;
  }
  for (int k = 0; k < n; ++k) {
    int rc = hold_sample(ctx, node_ids_host[k], R, B, cam_loc, ray_dirs, &poses[k], nullptr, factors[k].z_vals,
                         iters ? iters + k : nullptr, stream);
    if (rc) return rc;
    rc = hold_shade(ctx, node_ids_host[k], R, B, S, cam_loc, ray_dirs, &poses[k], &factors[k], stream);
    if (rc) return rc;
  }
  return hold_composite(ctx, n, R, S, factors, cls, comp, per_node, stream);
}

int hold_mesh_sdf(hold_ctx* ctx, int B, int P, const float* points, int V, const float* verts, int verts_batched, int F,
                  const int32_t* faces, float* sdf, int32_t* face_idx, void* stream) {
  HOLD_REQUIRE(ctx != nullptr, "ctx is NULL");
  HOLD_CUDA(cudaSetDevice(ctx->device));
  HOLD_REQUIRE(B >= 0 && P >= 0 && V > 0 && F > 0, "bad sizes");
  if (B == 0 || P == 0) return HOLD_OK;
  HOLD_REQUIRE(points && verts && faces && sdf, "NULL argument");
  dim3 grid(ceil_div(P, 128), B);
  k_mesh_sdf<<<grid, 128, 0, (cudaStream_t)stream>>>(P, V, F, verts_batched ? V * 3 : 0, points, verts, faces, sdf, face_idx);
  HOLD_LAUNCH_CHECK(ctx);
  return HOLD_OK;
}

int hold_off_in_surface(hold_ctx* ctx, int R, int S, const float* sdf, float threshold, uint8_t* off_surface,
                        uint8_t* in_surface, void* stream) {
  HOLD_REQUIRE(ctx != nullptr, "ctx is NULL");
  HOLD_CUDA(cudaSetDevice(ctx->device));
  HOLD_REQUIRE(R >= 0 && S >= 1, "bad sizes");
  if (R == 0) return HOLD_OK;
  HOLD_REQUIRE(sdf != nullptr, "NULL argument");
  k_off_in_surface<<<ceil_div(R, 128), 128, 0, (cudaStream_t)stream>>>(R, S, sdf, threshold, off_surface, in_surface);
  HOLD_LAUNCH_CHECK(ctx);
  return HOLD_OK;
}

int hold_inverse_warp_bwd(hold_ctx* ctx, int node, int B, int P, const float* x, const hold_node_pose* pose, const int32_t* knn_idx,
                          const float* g_xc, float* g_tfs, float* g_x, void* stream) {
  int rc = check_node(ctx, node, false);
  if (rc) return rc;
  HOLD_REQUIRE(B >= 0 && P >= 0, "bad sizes");
  if (B == 0) return HOLD_OK;
  HOLD_REQUIRE(pose && pose->tfs && g_tfs && (P == 0 || (x && g_xc)), "NULL argument");
  NodeState& ns = ctx->nodes[node];
  const bool hand = ns.cfg.kind == HOLD_KIND_HAND;
  cudaStream_t s = (cudaStream_t)stream;
  const int nb = max(1, ceil_div(P, 128));
  void* part = nullptr;
  if ((rc = ws_get(ctx, 22 /* WS_WARPBWD */, (size_t)B * nb * warpbwd::kJ * warpbwd::kG * sizeof(float), &part))) return rc;
  dim3 grid(nb, B);
  if (hand) {
    HOLD_REQUIRE(ns.has_rig, "hand node has no rig (hold_node_set_rig)");
    HOLD_REQUIRE(P == 0 || (knn_idx && pose->posed_verts), "hand backward needs the forward's knn_idx and the posed vertices");
    k_inverse_warp_bwd_hand<<<grid, 128, 0, s>>>(P, x, knn_idx, pose->posed_verts, ns.skin_w, pose->tfs, g_xc, g_x, (float*)part);
    HOLD_LAUNCH_CHECK(ctx);
    k_inverse_warp_bwd_hand_final<<<B, 256, 0, s>>>(nb, (const float*)part, g_tfs);
  } else {
    k_inverse_warp_bwd_obj<<<grid, 128, 0, s>>>(P, x, pose->tfs, g_xc, g_x, (float*)part);
    HOLD_LAUNCH_CHECK(ctx);
    k_inverse_warp_bwd_obj_final<<<B, 16, 0, s>>>(nb, (const float*)part, g_tfs);
  }
  HOLD_LAUNCH_CHECK(ctx);
  return HOLD_OK;
}

int hold_mise_destroy(hold_mise* h) {
  if (!h) return HOLD_OK;
  cudaFree(h->g.val), cudaFree(h->g.state), cudaFree(h->queue), cudaFree(h->counter);
  for (int L = 0; L < mise::kMaxDepth; ++L) { cudaFree(h->g.sub[L]); cudaFree(h->g.mark[L]); }
  delete h;
  return HOLD_OK;
}

int hold_mise_create(hold_ctx* ctx, int resolution_0, int depth, float threshold, hold_mise** out, void* stream) {
  HOLD_REQUIRE(ctx && out, "NULL argument");
  HOLD_CUDA(cudaSetDevice(ctx->device));
  HOLD_REQUIRE(resolution_0 >= 1 && depth >= 0 && depth <= mise::kMaxDepth, "bad MISE shape");
  HOLD_REQUIRE(((long long)resolution_0 << depth) <= 1024, "MISE resolution above 1024 is not supported");
  hold_mise* h = new (std::nothrow) hold_mise();
  HOLD_REQUIRE(h != nullptr, "out of host memory");
  h->ctx = ctx;
  mise::Grid& g = h->g;
  memset(&g, 0, sizeof(g));
  g.res0 = resolution_0, g.depth = depth, g.R = resolution_0 << depth, g.G = g.R + 1, g.threshold = threshold;
  h->np = (size_t)g.G * g.G * g.G;
  cudaStream_t s = (cudaStream_t)stream;
  cudaError_t e = cudaMalloc((void**)&g.val, h->np * sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc((void**)&g.state, h->np);
  if (e == cudaSuccess) e = cudaMalloc((void**)&h->queue, h->np * sizeof(int));
  if (e == cudaSuccess) e = cudaMalloc((void**)&h->counter, sizeof(unsigned int));
  for (int L = 0; L < depth && e == cudaSuccess; ++L) {
    const size_t n = (size_t)(resolution_0 << L) * (resolution_0 << L) * (resolution_0 << L);
    e = cudaMalloc((void**)&g.sub[L], n);
    if (e == cudaSuccess) e = cudaMalloc((void**)&g.mark[L], n * sizeof(unsigned int));
    if (e == cudaSuccess) e = cudaMemsetAsync(g.sub[L], 0, n, s);
  }
  if (e == cudaSuccess) e = cudaMemsetAsync(g.val, 0, h->np * sizeof(float), s);
  if (e == cudaSuccess) e = cudaMemsetAsync(g.state, 0, h->np, s);
  if (e != cudaSuccess) {
    set_error("hold_mise_create: %s", cudaGetErrorString(e));
    hold_mise_destroy(h);
    return HOLD_E_CUDA;
  }
  const int n0 = (resolution_0 + 1) * (resolution_0 + 1) * (resolution_0 + 1);
  k_mise_init<<<ceil_div(n0, 256), 256, 0, s>>>(g);
  HOLD_LAUNCH_CHECK(ctx);
  *out = h;
  return HOLD_OK;
}

int hold_mise_query(hold_mise* h, int32_t* coords, int capacity, int* n_points, void* stream) {
  HOLD_REQUIRE(h && n_points, "NULL argument");
  HOLD_CUDA(cudaSetDevice(h->ctx->device));
  cudaStream_t s = (cudaStream_t)stream;
  HOLD_CUDA(cudaMemsetAsync(h->counter, 0, sizeof(unsigned int), s));
  k_mise_collect<<<h->ctx->sm_count * 8, 256, 0, s>>>(h->g, h->queue, h->counter, (unsigned int)h->np);
  HOLD_LAUNCH_CHECK(h->ctx);
  unsigned int n = 0;
  HOLD_CUDA(cudaMemcpyAsync(&n, h->counter, sizeof(n), cudaMemcpyDeviceToHost, s));
  HOLD_CUDA(cudaStreamSynchronize(s));   // the caller sizes its SDF query by n: one host sync per MISE round, as in the reference loop
  h->n_last = (int)n;
  *n_points = (int)n;
  if (n == 0 || coords == nullptr) return HOLD_OK;
  HOLD_REQUIRE(capacity >= (int)n, "coords buffer holds %d points, %u needed", capacity, n);
  k_mise_coords<<<ceil_div((int)n, 256), 256, 0, s>>>(h->g, h->queue, (int)n, coords);
  HOLD_LAUNCH_CHECK(h->ctx);
  return HOLD_OK;
}

int hold_mise_update(hold_mise* h, const float* values, int n_values, void* stream) {
  HOLD_REQUIRE(h && (values || n_values == 0), "NULL argument");
  HOLD_CUDA(cudaSetDevice(h->ctx->device));
  HOLD_REQUIRE(n_values == h->n_last, "update with %d values after a query of %d points", n_values, h->n_last);
  cudaStream_t s = (cudaStream_t)stream;
  if (n_values > 0) {
    k_mise_scatter<<<ceil_div(n_values, 256), 256, 0, s>>>(h->g, h->queue, n_values, values);
    HOLD_LAUNCH_CHECK(h->ctx);
  }
  h->n_last = 0;
  const mise::Grid& g = h->g;
  for (int L = 0; L < g.depth; ++L) {
    const size_t n = (size_t)(g.res0 << L) * (g.res0 << L) * (g.res0 << L);
    HOLD_CUDA(cudaMemsetAsync(g.mark[L], 0, n * sizeof(unsigned int), s));
  }
  if (g.depth == 0) return HOLD_OK;
  k_mise_mark<<<h->ctx->sm_count * 8, 256, 0, s>>>(g);
  HOLD_LAUNCH_CHECK(h->ctx);
  for (int L = 0; L < g.depth; ++L) {
    k_mise_subdivide<<<h->ctx->sm_count * 4, 256, 0, s>>>(g, L);
    HOLD_LAUNCH_CHECK(h->ctx);
  }
  return HOLD_OK;
}

int hold_mise_to_dense(hold_mise* h, float* out, void* stream) {
  HOLD_REQUIRE(h && out, "NULL argument");
  HOLD_CUDA(cudaSetDevice(h->ctx->device));
  cudaStream_t s = (cudaStream_t)stream;
  k_mise_dense_init<<<h->ctx->sm_count * 8, 256, 0, s>>>(h->g, out);
  HOLD_LAUNCH_CHECK(h->ctx);
  for (int axis = 0; axis < 3; ++axis) {
    k_mise_fill<<<ceil_div(h->g.G * h->g.G, 128), 128, 0, s>>>(h->g, out, axis);
    HOLD_LAUNCH_CHECK(h->ctx);
  }
  return HOLD_OK;
}

/* ---- marching cubes on a dense value grid (SURVEY §8f rank 4: the last step of generate_mesh, utils/meshing.py:51) ---- */
int hold_mc_mark(hold_ctx* ctx, int n0, int n1, int n2, const float* vol, float level, int32_t* edge_flags, int32_t* cell_ntri, void* stream) {
  HOLD_REQUIRE(ctx && vol && edge_flags && cell_ntri, "NULL argument");
  HOLD_REQUIRE(n0 >= 2 && n1 >= 2 && n2 >= 2, "grid must be at least 2 x 2 x 2");
  HOLD_CUDA(cudaSetDevice(ctx->device));
  mc::Dims d{n0, n1, n2};
  const int64_t total = (int64_t)n0 * n1 * n2;
  k_mc_mark<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(d, vol, level, edge_flags, cell_ntri);
  HOLD_LAUNCH_CHECK(ctx);
  return HOLD_OK;
}

int hold_mc_emit(hold_ctx* ctx, int n0, int n1, int n2, const float* vol, float level, const int32_t* edge_flags, const int64_t* edge_vid,
                 const int64_t* cell_off, float* verts, int32_t* faces, void* stream) {
  HOLD_REQUIRE(ctx && vol && edge_flags && edge_vid && cell_off, "NULL argument");
  HOLD_REQUIRE(n0 >= 2 && n1 >= 2 && n2 >= 2, "grid must be at least 2 x 2 x 2");
  HOLD_CUDA(cudaSetDevice(ctx->device));
  mc::Dims d{n0, n1, n2};
  const int64_t total = (int64_t)n0 * n1 * n2;
  k_mc_emit<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(d, vol, level, edge_flags, edge_vid, cell_off, verts, faces);
  HOLD_LAUNCH_CHECK(ctx);
  return HOLD_OK;
}

/* measurement hook (not in the public header): key 2 = accumulator compensation c of the tcgen05 SDF chains (profiles/r02_tc_accumulator_bias.md) */
int hold_debug_set(hold_ctx* ctx, int key, int value) {
  if (!ctx) return HOLD_E_BADARG;
  if (key == 2) ctx->tc_acc_comp = value;
  else if (key == 3) ctx->sampler_passes = value;
  else return HOLD_E_BADARG;
  return HOLD_OK;
}

/* debug/test hook (not in the public header): workspace slot pointers of the last call */
int hold_debug_ws_copy(hold_ctx* ctx, int slot, void* dst, size_t bytes) {
  if (!ctx || slot < 0 || slot >= 24 || ctx->ws[slot].bytes < bytes) return HOLD_E_BADARG;
  HOLD_CUDA(cudaDeviceSynchronize());
  HOLD_CUDA(cudaMemcpy(dst, ctx->ws[slot].p, bytes, cudaMemcpyDeviceToDevice));
  return HOLD_OK;
}

int hold_bg_set_weights(hold_ctx* ctx, const hold_mlp_weights* sdf, const hold_mlp_weights* rgb, int mlp_mode, void* stream) {
  HOLD_REQUIRE(ctx && sdf && rgb, "NULL argument");
  HOLD_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t s = (cudaStream_t)stream;
  HOLD_REQUIRE(sdf->n_layers == 9 && rgb->n_layers == 2, "background nets: 9 + 2 layers expected");
  HOLD_REQUIRE(sdf->in_dim[0] == kBgEmbed + kBgFrame, "bg lin0 in_dim %d, expected 116", sdf->in_dim[0]);
  HOLD_REQUIRE(rgb->in_dim[0] == kBgView + kBgFrame + kFeat && rgb->out_dim[0] == 128 && rgb->out_dim[1] == 3 && rgb->in_dim[1] == 128,
               "bg colour head must be 315 -> 128 -> 3");
  PackedMlp& m = ctx->bg_sdf;
  int rc;
  for (int l = 0; l < 9; ++l) {
    const int eo = (l == 3) ? kHidden - kBgEmbed : (l == 8 ? kFeat + 1 : kHidden), ei = (l == 0) ? kBgEmbed + kBgFrame : kHidden;
    HOLD_REQUIRE(sdf->out_dim[l] == eo && sdf->in_dim[l] == ei, "bg lin%d is %dx%d, expected %dx%d", l, sdf->out_dim[l], sdf->in_dim[l], eo, ei);
    HOLD_REQUIRE(sdf->weight_v[l] && sdf->bias[l], "bg lin%d has NULL tensors", l);
    const int K = ei, Kpad = round_up(K, kKC), N = (l == 3) ? kHidden - kBgEmbed : kHidden, row_off = (l == 8) ? 1 : 0;
    m.K[l] = K, m.N[l] = N, m.Kpad[l] = Kpad, m.Npad[l] = 256;
    if ((rc = dev_alloc(&m.Wt[l], (size_t)Kpad * 256))) return rc;
    if ((rc = dev_alloc(&m.bias[l], 256))) return rc;
    const float scale = (l == 4) ? (float)(1.0 / sqrt(2.0)) : 1.0f;
    k_pack_layer<<<256, 128, 0, s>>>(sdf->weight_v[l], sdf->weight_g[l], sdf->bias[l], sdf->in_dim[l], row_off, 0, K, N, Kpad, scale, m.Wt[l], m.bias[l]);
    HOLD_LAUNCH_CHECK(ctx);
  }
  m.n_layers = 9;
  if ((rc = dev_alloc(&m.w_last, 256))) return rc;
  if ((rc = dev_alloc(&m.b_last, 4))) return rc;
  k_pack_rows<<<1, 128, 0, s>>>(sdf->weight_v[8], sdf->weight_g[8], sdf->bias[8], 256, 0, 1, m.w_last, m.b_last);
  HOLD_LAUNCH_CHECK(ctx);
  PackedMlp& c = ctx->bg_rgb;
  const int K0 = kBgView + kBgFrame + kFeat, K0pad = round_up(K0, kKC);
  c.K[0] = K0, c.N[0] = 128, c.Kpad[0] = K0pad, c.Npad[0] = 256;
  if ((rc = dev_alloc(&c.Wt[0], (size_t)K0pad * 256))) return rc;
  if ((rc = dev_alloc(&c.bias[0], 256))) return rc;
  k_pack_layer<<<256, 128, 0, s>>>(rgb->weight_v[0], rgb->weight_g[0], rgb->bias[0], K0, 0, 0, K0, 128, K0pad, 1.0f, c.Wt[0], c.bias[0]);
  HOLD_LAUNCH_CHECK(ctx);
  c.n_layers = 2;
  if ((rc = dev_alloc(&c.w_last, 3 * 128))) return rc;
  if ((rc = dev_alloc(&c.b_last, 4))) return rc;
  k_pack_rows<<<3, 128, 0, s>>>(rgb->weight_v[1], rgb->weight_g[1], rgb->bias[1], 128, 0, 3, c.w_last, c.b_last);
  HOLD_LAUNCH_CHECK(ctx);
  HOLD_REQUIRE(mlp_mode == HOLD_MLP_FP32 || mlp_mode == HOLD_MLP_TC, "bad mlp_mode");
  ctx->bg_mlp_mode = mlp_mode;
  if (mlp_mode == HOLD_MLP_TC && (rc = tc_bg_pack(ctx, ctx->bg_tc, sdf, rgb, s))) return rc;
  ctx->has_bg = true;
  return HOLD_OK;
}

int hold_background(hold_ctx* ctx, int R, int B, const float* cam_loc, const float* ray_dirs, const float* frame_code,
                    const float* fg_bg_weights, float* bg_rgb, float* bg_rgb_only, float* bg_semantics, float* bg_z_vals,
                    void* stream) {
  HOLD_REQUIRE(ctx != nullptr, "ctx is NULL");
  HOLD_CUDA(cudaSetDevice(ctx->device));
  if (!ctx->has_bg) { set_error("background weights not set (hold_bg_set_weights)"); return HOLD_E_STATE; }
  HOLD_REQUIRE(R >= 0 && B >= 1, "bad R/B");
  if (R == 0) return HOLD_OK;
  HOLD_REQUIRE(R % B == 0, "R (%d) must be B (%d) frames x rays, frame-major", R, B);
  HOLD_REQUIRE(cam_loc && ray_dirs && frame_code && fg_bg_weights, "NULL argument");
  cudaStream_t s = (cudaStream_t)stream;
  const int rpf = R / B;
  const int rays_per_chunk = max(1, min(rpf, (1 << 20) / kBgN));
  const size_t cp = (size_t)rays_per_chunk * kBgN;
  WS(WS_BGSDF, float, cp, sdf_ws);
  WS(WS_BGFEAT, float, cp * kFeat, feat_ws);
  WS(WS_BGRGB, float, cp * 3, rgb_ws);
  for (int b = 0; b < B; ++b) {
    for (int r0 = 0; r0 < rpf; r0 += rays_per_chunk) {
      const int rn = min(rays_per_chunk, rpf - r0), P = rn * kBgN;
      const size_t ray0 = (size_t)b * rpf + r0;
      BgArgs a;
      memset(&a, 0, sizeof(a));
      a.P = P, a.pts_per_frame = P, a.cam = cam_loc + ray0 * 3, a.dirs = ray_dirs + ray0 * 3, a.frame_code = frame_code + (size_t)b * kBgFrame;
      a.r_sphere = 0.f;
      // the bounding sphere is a per-node constant in the reference (same value for all nodes): take node 0's
      for (int n = 0; n < HOLD_MAX_NODES; ++n)
        if (ctx->nodes[n].configured) { a.r_sphere = ctx->nodes[n].cfg.bounding_sphere; break; }
      HOLD_REQUIRE(a.r_sphere > 0.f, "configure a node first (scene_bounding_sphere)");
      a.n_layers = 9;
      for (int l = 0; l < 9; ++l) { a.L[l].Wt = ctx->bg_sdf.Wt[l], a.L[l].bias = ctx->bg_sdf.bias[l], a.L[l].Kpad = ctx->bg_sdf.Kpad[l], a.L[l].N = ctx->bg_sdf.N[l]; }
      a.w_last = ctx->bg_sdf.w_last, a.b_last = ctx->bg_sdf.b_last, a.sdf = sdf_ws, a.feat = feat_ws;
      if (ctx->bg_mlp_mode == HOLD_MLP_TC && ctx->bg_tc != nullptr) {
        int rc = tc_bg_launch(ctx, *ctx->bg_tc, P, a.cam, a.dirs, a.frame_code, a.r_sphere, sdf_ws, feat_ws, rgb_ws, s);
        if (rc) return rc;
      } else {
        const int tiles = ceil_div(P, kTileRows);
        k_bg_mlp<BG_SDF><<<min(tiles, ctx->sm_count), 256, kBgSmemBytes, s>>>(a);
        HOLD_LAUNCH_CHECK(ctx);
        BgArgs c = a;
        c.n_layers = 1;
        c.L[0].Wt = ctx->bg_rgb.Wt[0], c.L[0].bias = ctx->bg_rgb.bias[0], c.L[0].Kpad = ctx->bg_rgb.Kpad[0], c.L[0].N = 128;
        c.w_last = ctx->bg_rgb.w_last, c.b_last = ctx->bg_rgb.b_last, c.rgb = rgb_ws;
        k_bg_mlp<BG_RGB><<<min(tiles, ctx->sm_count), 256, kBgSmemBytes, s>>>(c);
        HOLD_LAUNCH_CHECK(ctx);
      }
      k_bg_composite<<<ceil_div(rn, 128), 128, 0, s>>>(rn, a.r_sphere, sdf_ws, rgb_ws, fg_bg_weights + ray0,
                                                       bg_rgb ? bg_rgb + ray0 * 3 : nullptr, bg_rgb_only ? bg_rgb_only + ray0 * 3 : nullptr,
                                                       bg_semantics ? bg_semantics + ray0 * 4 : nullptr, bg_z_vals ? bg_z_vals + ray0 * kBgN : nullptr);
      HOLD_LAUNCH_CHECK(ctx);
    }
  }
  return HOLD_OK;
}

int hold_sdf_eval(hold_ctx* ctx, int node, int P, const float* x_c, const float* embed_w, float* sdf, float* grad,
                  float* feat, void* stream) {
  int rc = check_node(ctx, node, true);
  if (rc) return rc;
  HOLD_REQUIRE(P >= 0, "negative P");
  if (P == 0) return HOLD_OK;
  HOLD_REQUIRE(x_c && sdf, "NULL argument");
  HOLD_REQUIRE((grad == nullptr) == (feat == nullptr), "grad and feat must be requested together");
  return launch_sdf(ctx, ctx->nodes[node], P, x_c, embed_w, sdf, grad, feat, nullptr, (cudaStream_t)stream);
}

int hold_linear(hold_ctx* ctx, int node, int mat, int P, const float* A, int lda, int kvalid, int add_bias, const float* in_scale,
                float* C, int ldc, int nvalid, void* stream) {
  HOLD_REQUIRE(ctx != nullptr, "ctx is NULL");
  HOLD_REQUIRE(P >= 0, "negative P");
  if (P == 0) return HOLD_OK;
  HOLD_REQUIRE(A && C, "NULL argument");
  const uint8_t* img = nullptr;
  const float* bias = nullptr;
  int nst = 8, kmax = 256, nmax = 256;
  if (node == -1) {   // the background nets (hold_bg_set_weights with HOLD_MLP_TC)
    HOLD_CUDA(cudaSetDevice(ctx->device));
    HOLD_REQUIRE(ctx->has_bg && ctx->bg_tc != nullptr, "hold_linear(node -1) needs tensor-core background weights (hold_bg_set_weights, HOLD_MLP_TC)");
    const TcBg& t = *ctx->bg_tc;
    constexpr int kIn = kBgEmbed + kBgFrame;   // lin0: 116 inputs; the skip at layer 4 re-feeds the 84 embedding columns (lin3: 172 outputs)
    if (mat >= 0 && mat <= 8) { img = t.sdf_img[mat]; bias = ctx->bg_sdf.bias[mat]; nst = t.sdf_nst[mat]; kmax = (mat == 0) ? kIn : 256; nmax = (mat == 3) ? 256 - kBgEmbed : 256; }
    else if (mat >= 16 && mat <= 24) { img = t.sdf_imgT[mat - 16]; kmax = (mat == 19) ? 256 - kBgEmbed : 256; nmax = (mat == 16) ? kIn : 256; }
    else if (mat == 32) { img = t.rgb_img; bias = ctx->bg_rgb.bias[0]; nst = 10; kmax = 320; nmax = 128; }
    else if (mat == 48 || mat == 49) { img = t.rgb_imgT[mat - 48]; kmax = 128; nmax = (mat == 49) ? 64 : 256; }
  } else {
    int rc = check_node(ctx, node, true);
    if (rc) return rc;
    NodeState& ns = ctx->nodes[node];
    HOLD_REQUIRE(ns.tc != nullptr, "hold_linear needs the packed tcgen05 weight images (hold_node_set_weights)");
    if (mat >= 0 && mat <= 8) { img = ns.tc->sdf_img[mat]; bias = ns.sdf.bias[mat]; nst = ns.tc->sdf_nst[mat]; kmax = (mat == 0) ? kEmbed : 256; nmax = ns.sdf.N[mat]; }
    else if (mat >= 16 && mat <= 24) { img = ns.tc->sdf_imgT[mat - 16]; kmax = (mat - 16 == 3) ? kHidden - kEmbed : 256; nmax = (mat == 16) ? kEmbed : 256; }
    else if (mat >= 32 && mat <= 35) { img = ns.tc->rgb_img[mat - 32]; bias = ns.rgb.bias[mat - 32]; nst = ns.tc->rgb_nst[mat - 32]; kmax = (mat == 32) ? 320 : 256; }
    else if (mat >= 48 && mat <= 52) { img = ns.tc->rgb_imgT[mat - 48]; nmax = (mat == 49) ? 64 : 256; }
  }
  HOLD_REQUIRE(img != nullptr, "hold_linear: unknown matrix id %d for node %d", mat, node);
  HOLD_REQUIRE(kvalid >= 1 && kvalid <= kmax && nvalid >= 1 && nvalid <= nmax, "hold_linear(%d): kvalid %d (max %d) / nvalid %d (max %d)", mat, kvalid, kmax, nvalid, nmax);
  HOLD_REQUIRE(!add_bias || bias != nullptr, "hold_linear(%d): this matrix has no bias", mat);
  return tc_launch_linear_img(ctx, img, add_bias ? bias : nullptr, nst, P, A, lda, kvalid, in_scale, C, ldc, nvalid, (cudaStream_t)stream);
}

int hold_wgrad(hold_ctx* ctx, int P, const float* D, int ldd, int N, const float* A, int lda, int K, const float* d_scale,
               const float* a_scale, float* out, int ldo, void* stream) {
  HOLD_REQUIRE(ctx && D && A && out, "NULL argument");
  HOLD_REQUIRE(P >= 0 && N >= 1 && N <= 256 && K >= 1 && K <= 256 && ldd >= N && lda >= K && ldo >= K, "hold_wgrad: N, K in [1, 256]");
  HOLD_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t s = (cudaStream_t)stream;
  HOLD_CUDA(cudaMemset2DAsync(out, (size_t)ldo * sizeof(float), 0, (size_t)K * sizeof(float), N, s));
  if (P == 0) return HOLD_OK;
  WgArgs a;
  a.P = P, a.N = N, a.K = K, a.ldd = ldd, a.lda = lda, a.ldo = ldo, a.D = D, a.A = A, a.d_scale = d_scale, a.a_scale = a_scale;
  a.out = out, a.err = ctx->dev_err;
  const int slabs = ceil_div(P, kWgPts);
  k_wgrad_tc<<<min(slabs, ctx->sm_count), kWgThreads, kWgSmem, s>>>(a);
  HOLD_LAUNCH_CHECK(ctx);
  return HOLD_OK;
}

int hold_pow2_scale(hold_ctx* ctx, int P, int ncols, const float* x, int ld, float* scale_out, void* stream) {
  HOLD_REQUIRE(ctx && x && scale_out, "NULL argument");
  HOLD_REQUIRE(P >= 1 && ncols >= 1 && ld >= ncols, "bad sizes");
  HOLD_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t s = (cudaStream_t)stream;
  void* w = nullptr;
  int rc = ws_get(ctx, 21 /* WS_AMAX */, 256, &w);
  if (rc) return rc;
  // one word per call, rotating through the workspace so that back-to-back calls on a stream never share a counter in flight
  unsigned int* bits = (unsigned int*)w + (ctx->launches & 31);
  HOLD_CUDA(cudaMemsetAsync(bits, 0, sizeof(unsigned int), s));
  const size_t total = (size_t)P * ncols;
  k_absmax_bits<<<(int)std::min<size_t>((total + 255) / 256, (size_t)ctx->sm_count * 8), 256, 0, s>>>(P, ncols, x, ld, bits);
  HOLD_LAUNCH_CHECK(ctx);
  k_pow2_scale<<<1, 1, 0, s>>>(bits, scale_out);
  HOLD_LAUNCH_CHECK(ctx);
  return HOLD_OK;
}

int hold_train_ew(hold_ctx* ctx, int op, int P, const hold_ew_args* args, void* stream) {
  HOLD_REQUIRE(ctx && args, "NULL argument");
  HOLD_REQUIRE(op >= 0 && op <= EW_RELU_BWD && P >= 0, "bad op / P");
  if (P == 0) return HOLD_OK;
  HOLD_CUDA(cudaSetDevice(ctx->device));
  EwArgs a;
  a.in0 = args->in0, a.in1 = args->in1, a.in2 = args->in2, a.out0 = args->out0, a.out1 = args->out1;
  a.ld_in0 = args->ld_in0, a.ld_in1 = args->ld_in1, a.ld_in2 = args->ld_in2, a.ld_out0 = args->ld_out0, a.ld_out1 = args->ld_out1;
  a.ncols = args->ncols, a.aux = args->aux;
  HOLD_REQUIRE(a.ncols >= 1 && a.ncols <= 320 && a.in0 && a.out0, "bad elementwise arguments");
  const size_t total = (size_t)P * (size_t)a.ncols;
  const int blocks = (int)std::min<size_t>((total + 255) / 256, (size_t)ctx->sm_count * 16);
  k_train_ew<<<blocks, 256, 0, (cudaStream_t)stream>>>(op, P, a);
  HOLD_LAUNCH_CHECK(ctx);
  return HOLD_OK;
}

int hold_rgb_eval(hold_ctx* ctx, int node, int B, int P, const float* x_c, const float* normals, const float* pose_cond,
                  const float* feat, const float* time_code, float* rgb, void* stream) {
  int rc = check_node(ctx, node, true);
  if (rc) return rc;
  HOLD_REQUIRE(B >= 1 && P >= 0, "bad sizes");
  if (P == 0) return HOLD_OK;
  HOLD_REQUIRE(P % B == 0, "P (%d) must be B (%d) frames x points, frame-major", P, B);
  HOLD_REQUIRE(x_c && normals && feat && rgb, "NULL argument");
  NodeState& ns = ctx->nodes[node];
  const bool hand = ns.cfg.kind == HOLD_KIND_HAND;
  cudaStream_t s = (cudaStream_t)stream;
  float* pe = nullptr;
  if (hand) {
    HOLD_REQUIRE(pose_cond != nullptr, "hand node needs pose_cond [B,45] (zeros give lin_pose's bias, texture_net.py:80-82)");
    WS(WS_PE, float, (size_t)B * 8, pe_ws);
    pe = pe_ws;
    k_pose_embed<<<ceil_div(B * 8, 64), 64, 0, s>>>(B, pose_cond, ns.lin_pose_w, ns.lin_pose_b, pe);
    HOLD_LAUNCH_CHECK(ctx);
  } else {
    HOLD_REQUIRE(time_code != nullptr, "object node needs time_code [B,32]");
  }
  return launch_rgb(ctx, ns, P, P / B, x_c, normals, pe, feat, hand ? nullptr : time_code, rgb, s);
}

int hold_forward_warp(hold_ctx* ctx, int node, int B, int P, const float* x_c, const hold_node_pose* pose, float* x_d,
                      int32_t* knn_idx, uint8_t* outlier_mask, void* stream) {
  int rc = check_node(ctx, node, false);
  if (rc) return rc;
  HOLD_REQUIRE(B >= 0 && P >= 0, "negative size");
  if (B * P == 0) return HOLD_OK;
  HOLD_REQUIRE(x_c && pose && x_d && pose->tfs, "NULL argument");
  NodeState& ns = ctx->nodes[node];
  dim3 grid(ceil_div(P, 128), B);
  cudaStream_t s = (cudaStream_t)stream;
  if (ns.cfg.kind == HOLD_KIND_HAND) {
    if (!ns.has_rig) { set_error("hand node has no rig (hold_node_set_rig)"); return HOLD_E_STATE; }
    k_inverse_warp<true, false, true><<<grid, 128, 0, s>>>(P, 1, 1, nullptr, nullptr, nullptr, x_c, pose->tfs, ns.cano_verts, ns.skin_w, x_d,
                                                           knn_idx, outlier_mask, nullptr, ctx->dev_err);
  } else {
    k_inverse_warp<false, false, true><<<grid, 128, 0, s>>>(P, 1, 1, nullptr, nullptr, nullptr, x_c, pose->tfs, nullptr, nullptr, x_d,
                                                            nullptr, nullptr, nullptr, ctx->dev_err);
  }
  HOLD_LAUNCH_CHECK(ctx);
  return HOLD_OK;
}

int hold_inverse_warp(hold_ctx* ctx, int node, int B, int P, const float* x, const hold_node_pose* pose, float* x_c,
                      int32_t* knn_idx, uint8_t* outlier_mask, void* stream) {
  int rc = check_node(ctx, node, false);
  if (rc) return rc;
  HOLD_REQUIRE(B >= 0 && P >= 0, "negative size");
  if (B * P == 0) return HOLD_OK;
  HOLD_REQUIRE(x && pose && x_c && pose->tfs, "NULL argument");
  return launch_inverse_warp(ctx, ctx->nodes[node], B, P, false, 1, 1, nullptr, nullptr, nullptr, x, pose, x_c, knn_idx,
                             outlier_mask, nullptr, (cudaStream_t)stream);
}

// ------------------------------------------------------------------------------------------------ training glue (train_glue.cuh)
static int nd_blocks(int P) { return max(1, ceil_div(P, kGlueThreads)); }

int hold_train_glue_sizes(hold_ctx* ctx, int node, int B, int P, int64_t* stash_floats, int64_t* scratch_floats) {
  int rc = check_node(ctx, node, false);
  if (rc) return rc;
  HOLD_REQUIRE(B >= 0 && P >= 0, "negative size");
  const bool hand = ctx->nodes[node].cfg.kind == HOLD_KIND_HAND;
  if (stash_floats) *stash_floats = (int64_t)B * P * (hand ? glue::kStashHand : glue::kStashObj);
  if (scratch_floats) *scratch_floats = (int64_t)B * nd_blocks(P) * (hand ? glue::kPartHand : glue::kPartObj);
  return HOLD_OK;
}

int hold_normal_density(hold_ctx* ctx, int node, int B, int P, const float* x_c, const float* grad, const float* sdf,
                        const float* tfs, const float* beta, float* normal, float* density, float* stash, void* stream) {
  int rc = check_node(ctx, node, false);
  if (rc) return rc;
  HOLD_REQUIRE(B >= 0 && P >= 0, "negative size");
  if (B * P == 0) return HOLD_OK;
  HOLD_REQUIRE(grad && sdf && tfs && beta && normal && density && stash, "NULL argument");
  NodeState& ns = ctx->nodes[node];
  const bool hand = ns.cfg.kind == HOLD_KIND_HAND;
  dim3 grid(nd_blocks(P), B);
  cudaStream_t s = (cudaStream_t)stream;
  if (hand) {
    HOLD_REQUIRE(ns.has_rig, "hand node has no rig (hold_node_set_rig)");
    HOLD_REQUIRE(x_c != nullptr, "hand node needs x_c for the skinning weights");
    k_nd_fwd<true><<<grid, kGlueThreads, 0, s>>>(P, x_c, grad, sdf, tfs, ns.cano_verts, ns.skin_w, beta, normal, density, stash);
  } else {
    k_nd_fwd<false><<<grid, kGlueThreads, 0, s>>>(P, x_c, grad, sdf, tfs, nullptr, nullptr, beta, normal, density, stash);
  }
  HOLD_LAUNCH_CHECK(ctx);
  return HOLD_OK;
}

int hold_normal_density_bwd(hold_ctx* ctx, int node, int B, int P, const float* grad, const float* sdf, const float* beta,
                            const float* stash, const float* d_normal, const float* d_density, float* d_grad, float* d_sdf,
                            float* d_tfs, float* d_beta, float* scratch, void* stream) {
  int rc = check_node(ctx, node, false);
  if (rc) return rc;
  HOLD_REQUIRE(B >= 0 && P >= 0, "negative size");
  if (B == 0) return HOLD_OK;
  HOLD_REQUIRE(beta && d_tfs && d_beta && scratch, "NULL argument");
  HOLD_REQUIRE(P == 0 || (grad && sdf && stash && d_grad && d_sdf), "NULL argument");
  const bool hand = ctx->nodes[node].cfg.kind == HOLD_KIND_HAND;
  const int nb = nd_blocks(P);
  dim3 grid(nb, B);
  cudaStream_t s = (cudaStream_t)stream;
  if (hand) {
    k_nd_bwd<true><<<grid, kGlueThreads, 0, s>>>(P, grad, sdf, beta, stash, d_normal, d_density, d_grad, d_sdf, scratch);
    HOLD_LAUNCH_CHECK(ctx);
    k_nd_bwd_final<true><<<B, 256, 0, s>>>(nb, scratch, d_tfs, d_beta);
  } else {
    k_nd_bwd<false><<<grid, kGlueThreads, 0, s>>>(P, grad, sdf, beta, stash, d_normal, d_density, d_grad, d_sdf, scratch);
    HOLD_LAUNCH_CHECK(ctx);
    k_nd_bwd_final<false><<<B, 16, 0, s>>>(nb, scratch, d_tfs, d_beta);
  }
  HOLD_LAUNCH_CHECK(ctx);
  return HOLD_OK;
}

int hold_bg_inputs(hold_ctx* ctx, int R, float r_sphere, const float* cam_loc, const float* ray_dirs, float* emb_pts,
                   float* emb_view, void* stream) {
  HOLD_REQUIRE(ctx != nullptr, "ctx is NULL");
  HOLD_REQUIRE(R >= 0 && r_sphere > 0.f, "bad R / r_sphere");
  if (R == 0) return HOLD_OK;
  HOLD_REQUIRE(cam_loc && ray_dirs && emb_pts && emb_view, "NULL argument");
  HOLD_CUDA(cudaSetDevice(ctx->device));
  k_bg_inputs<<<ceil_div(R * kBgN, kGlueThreads), kGlueThreads, 0, (cudaStream_t)stream>>>(R, r_sphere, cam_loc, ray_dirs, emb_pts, emb_view);
  HOLD_LAUNCH_CHECK(ctx);
  return HOLD_OK;
}

int hold_bg_integrate(hold_ctx* ctx, int R, float r_sphere, const float* sdf, int ld_sdf, const float* rgb, const float* fg_bg_weights,
                      float* bg_rgb, float* bg_rgb_only, float* bg_semantics, void* stream) {
  HOLD_REQUIRE(ctx != nullptr, "ctx is NULL");
  HOLD_REQUIRE(R >= 0 && r_sphere > 0.f && ld_sdf >= 1, "bad R / r_sphere / ld_sdf");
  if (R == 0) return HOLD_OK;
  HOLD_REQUIRE(sdf && rgb && fg_bg_weights, "NULL argument");
  HOLD_CUDA(cudaSetDevice(ctx->device));
  k_bg_integrate<<<ceil_div(R, kGlueThreads), kGlueThreads, 0, (cudaStream_t)stream>>>(R, r_sphere, sdf, ld_sdf, rgb, fg_bg_weights, bg_rgb,
                                                                                    bg_rgb_only, bg_semantics);
  HOLD_LAUNCH_CHECK(ctx);
  return HOLD_OK;
}

int hold_bg_integrate_bwd(hold_ctx* ctx, int R, float r_sphere, const float* sdf, int ld_sdf, const float* rgb,
                          const float* fg_bg_weights, const float* g_bg_rgb, const float* g_bg_rgb_only, const float* g_bg_semantics,
                          float* d_rgb, float* d_sdf, float* d_fg_bg_weights, void* stream) {
  HOLD_REQUIRE(ctx != nullptr, "ctx is NULL");
  HOLD_REQUIRE(R >= 0 && r_sphere > 0.f && ld_sdf >= 1, "bad R / r_sphere / ld_sdf");
  if (R == 0) return HOLD_OK;
  HOLD_REQUIRE(sdf && rgb && fg_bg_weights && d_rgb && d_sdf && d_fg_bg_weights, "NULL argument");
  HOLD_CUDA(cudaSetDevice(ctx->device));
  k_bg_integrate_bwd<<<ceil_div(R, kGlueThreads), kGlueThreads, 0, (cudaStream_t)stream>>>(R, r_sphere, sdf, ld_sdf, rgb, fg_bg_weights, g_bg_rgb,
                                                                                        g_bg_rgb_only, g_bg_semantics, d_rgb, d_sdf, d_fg_bg_weights);
  HOLD_LAUNCH_CHECK(ctx);
  return HOLD_OK;
}

}  // extern "C"
