/* hold_b200 — C ABI of the B200-native HOLD volumetric-rendering hot path.
 *
 * The reference (zc-alexfan/hold) has no FFI/plugin layer: its call surface for this path is a set of
 * Python classes (SURVEY.md §8b).  Each entry point below replaces the body of one of them; the
 * reference-side binding (a ctypes stub inside the unchanged Python class) is shown in INTEGRATION.md.
 * All file:line citations are relative to /root/reference/code/src.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer to contiguous row-major fp32 unless the name ends in `_host`
 *    or the comment says otherwise; integer outputs are int32;
 *  - every call enqueues on `stream` (a cudaStream_t passed as void*) and never synchronises the host —
 *    including the sampler's batch-global convergence flag (engine/ray_sampler.py:244);
 *  - the caller owns all input/output buffers; the library owns only its workspace and packed weights;
 *  - return value: 0 on success, a negative hold_status otherwise; text via hold_last_error();
 *  - never exit()/abort (contrast engine/ray_sampler.py:16-18).
 */
#ifndef HOLD_B200_H
#define HOLD_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HOLD_B200_VERSION 200 /* major*10000 + minor*100 + patch */

typedef enum hold_status {
  HOLD_OK = 0,
  HOLD_E_BADARG = -1,
  HOLD_E_CUDA = -2,
  HOLD_E_RAY_MISSES_SPHERE = -3, /* reported by hold_ctx_check(), engine/ray_sampler.py:15-18 */
  HOLD_E_NONFINITE = -4,
  HOLD_E_NOMEM = -5,
  HOLD_E_STATE = -6
} hold_status;

typedef struct hold_ctx hold_ctx;

enum { HOLD_KIND_HAND = 0, HOLD_KIND_OBJECT = 1 };
/* MLP arithmetic: exact fp32 on CUDA cores, or tcgen05 with fp16 hi/lo split operands, 3 passes (fp32 accumulate). */
enum { HOLD_MLP_FP32 = 0, HOLD_MLP_TC = 1 };
enum { HOLD_MAX_NODES = 4, HOLD_MAX_LAYERS = 9 };

/* Node.__init__ + confs/general.yaml `ray_sampler`/`implicit_network` constants
 * (model/renderables/node.py:17-47; engine/ray_sampler.py:89-126). */
typedef struct hold_node_cfg {
  int32_t kind;            /* HOLD_KIND_* */
  int32_t class_id;        /* semantics channel: object 1, right 2, left 3 (engine/rendering.py:59-61) */
  int32_t n_samples_eval;  /* N_samples_eval (128) */
  int32_t n_samples;       /* N_samples (64) */
  int32_t n_samples_extra; /* N_samples_extra (32) */
  int32_t beta_iters;      /* 10 */
  int32_t max_total_iters; /* 5 */
  int32_t mlp_mode;        /* HOLD_MLP_* */
  float eps;               /* 0.1 */
  float add_tiny;          /* 1e-6 */
  float near;              /* 0.0 */
  float bounding_sphere;   /* scene_bounding_sphere */
  float beta_min;          /* LaplaceDensity beta_min, 1e-4 (engine/density.py:17-19) */
} hold_node_cfg;

/* One MLP in the reference's state_dict layout: lin<k>.weight_v [out,in], lin<k>.weight_g [out,1],
 * lin<k>.bias [out] (networks/shape_net.py:79-81, texture_net.py:39-41).  weight_g may be NULL for a
 * layer without weight-norm (then weight_v is the plain weight). */
typedef struct hold_mlp_weights {
  int32_t n_layers;
  int32_t in_dim[HOLD_MAX_LAYERS];
  int32_t out_dim[HOLD_MAX_LAYERS];
  const float* weight_v[HOLD_MAX_LAYERS];
  const float* weight_g[HOLD_MAX_LAYERS];
  const float* bias[HOLD_MAX_LAYERS];
} hold_mlp_weights;

/* MANO model tensors (utils/external/body_models.py:502-560; lbs() arguments utils/external/lbs.py:139-151). */
typedef struct hold_mano_model {
  const float* v_template;  /* [778,3] */
  const float* shapedirs;   /* [778,3,10] */
  const float* posedirs;    /* [135,2334] */
  const float* J_regressor; /* [16,778] */
  const float* lbs_weights; /* [778,16] */
  const float* hands_mean;  /* [45] (pose_mean = [0,0,0,hands_mean], flat_hand_mean=False) */
  const int32_t* parents_host; /* [16] HOST pointer, parents[0] = -1 */
  const int32_t* tip_ids_host; /* [5]  HOST pointer (vertex_ids 'mano') */
} hold_mano_model;

/* Per-call articulation of one node, as produced by the servers (a16/a17). */
typedef struct hold_node_pose {
  const float* tfs;         /* hand: [B,16,4,4] (relative to canonical); object: [B,4,4] */
  const float* posed_verts; /* hand: [B,778,3] (deform_info["verts"]); object: NULL */
  const float* pose_cond;   /* hand: [B,45] = full_pose[:,3:]/pi (or zeros), object: NULL */
  const float* time_code;   /* object: [B,32] frame latent; hand: NULL */
  const float* embed_w;     /* [39] BARF weights or NULL (plain Fourier) */
  const float* beta_param;  /* [1] density.beta parameter (device scalar) */
} hold_node_pose;

/* Outputs of Node.forward (`factors`, model/renderables/node.py:78-86) for R rays x S samples. */
typedef struct hold_factors {
  float* color;         /* [R,S,3] */
  float* normal;        /* [R,S,3] */
  float* density;       /* [R,S]   */
  float* z_vals;        /* [R,S]   */
  float* sdf;           /* [R,S]   optional (may be NULL) */
  float* canonical_pts; /* [R,S,3] optional */
} hold_factors;

/* Outputs of volumetric_render (hold/hold_utils.py:243-271). Any pointer may be NULL to skip it. */
typedef struct hold_render_out {
  float* fg_rgb;       /* [R,3] */
  float* mask_prob;    /* [R]   */
  float* normal;       /* [R,3] */
  float* depth;        /* [R]   */
  float* fg_semantics; /* [R,4] */
  float* bg_weights;   /* [R]   */
  float* fg_weights;   /* [R,S_out] */
} hold_render_out;

/* Training-mode randomness is an INPUT (generated by torch on the host side of the boundary):
 * stratified jitter (ray_sampler.py:70-78), u (:292), extras permutation (:328).  All NULL in eval.
 * The reference draws the extras as randperm(n)[:N_extra] with n = the size of the z buffer when the loop ends, i.e.
 * rounds * N_eval — known only on the device.  The caller therefore supplies one draw per possible round count:
 * extra_idx[j] = randperm((j + 1) * N_eval)[:N_extra]; the kernels use row (rounds - 1). */
typedef struct hold_sampler_rand {
  const float* jitter;      /* [R, n_samples_eval] uniforms */
  const float* u;           /* [R, n_samples] uniforms */
  const int32_t* extra_idx; /* [max_total_iters, n_samples_extra] indices into the final z buffer, one row per round count */
} hold_sampler_rand;

int hold_version(void);
const char* hold_last_error(void); /* thread-local */
int hold_ctx_create(hold_ctx** out, int device);
int hold_ctx_destroy(hold_ctx* ctx);
/* Synchronises `stream` and reads the device error word (ray missed the bounding sphere, non-finite). */
int hold_ctx_check(hold_ctx* ctx, void* stream);
/* Number of kernels this library launched since the ctx was created (bench.py's gpu_launches). */
int64_t hold_ctx_launch_count(hold_ctx* ctx);

int hold_node_configure(hold_ctx* ctx, int node, const hold_node_cfg* cfg);
/* Fold weight-norm (shape_net.py:80), drop the hand's 45 zeroed pose columns (shape_net.py:104-106),
 * pre-scale the skip layer by 1/sqrt(2) (shape_net.py:122), pack for both MLP modes.  Re-call after
 * every optimiser step / load_state_dict.  lin_pose_* : RenderingNet.lin_pose (texture_net.py:32-37). */
int hold_node_set_weights(hold_ctx* ctx, int node, const hold_mlp_weights* sdf, const hold_mlp_weights* rgb,
                          const float* lin_pose_w, const float* lin_pose_b, void* stream);
/* Canonical rig of a hand node: KNNDeformer.verts / .skin_weights (model/mano/deformer.py:17-32). */
int hold_node_set_rig(hold_ctx* ctx, int node, const float* cano_verts /*[778,3]*/,
                      const float* skin_weights /*[778,16]*/, void* stream);

/* a16: GenericServer.forward (model/mano/server.py:62-99) = MANO lbs() + scene scaling + tfs_c_inv.
 * tfs_c_inv NULL <=> absolute=True.  Outputs: verts [B,778,3], jnts [B,21,3], tfs [B,16,4,4], v_posed [B,778,3]. */
int hold_mano_lbs(hold_ctx* ctx, const hold_mano_model* m, int B, const float* betas /*[B,10]*/,
                  const float* full_pose /*[B,48]*/, const float* transl /*[B,3]*/, const float* scene_scale /*[B]*/,
                  const float* tfs_c_inv /*[16,4,4] or NULL*/, float* verts, float* jnts, float* tfs, float* v_posed,
                  void* stream);
/* Reverse mode of hold_mano_lbs — what torch.autograd computes through GenericServer.forward for the pose refinement
 * of optimize_ckpt.py (fitting/model.py:117; SURVEY §8f rank 4).  Upstream gradients g_verts [B,778,3], g_jnts [B,21,3],
 * g_tfs [B,16,4,4] (each may be NULL = zero) -> g_betas [B,10], g_pose [B,48], g_transl [B,3], g_scale [B].
 * Deterministic (fixed-order sums). */
int hold_mano_lbs_bwd(hold_ctx* ctx, const hold_mano_model* m, int B, const float* betas, const float* full_pose,
                      const float* transl, const float* scene_scale, const float* tfs_c_inv, const float* g_verts,
                      const float* g_jnts, const float* g_tfs, float* g_betas, float* g_pose, float* g_transl, float* g_scale,
                      void* stream);
/* Reverse mode of hold_object_tf (ObjectModel.forward under autograd).  g_verts [B,Nv,3], g_tfs [B,4,4] (nullable) ->
 * g_rot [B,3], g_trans [B,3], g_scene_scale [B], g_obj_scale [B] (per-frame terms of the scalar's gradient). */
int hold_object_tf_bwd(hold_ctx* ctx, int B, const float* rot, const float* trans, const float* scene_scale, float obj_scale,
                       const float* denorm_mat, const float* pts_cano, int Nv, const float* g_verts, const float* g_tfs,
                       float* g_rot, float* g_trans, float* g_scene_scale, float* g_obj_scale, void* stream);
/* Training-only loss targets (SURVEY §8f rank 3) — replaces the reference's kaolin v0.10.0 calls in
 * compute_mano_cano_sdf / check_off_in_surface_points_cano_mesh (engine/volsdf_utils.py:172-217):
 * sdf[b,p] = sqrt(point_to_mesh_distance) * (1 - 2 * check_sign) of points [B,P,3] against the closed mesh
 * (verts [B,V,3] if verts_batched else [V,3] shared by all frames; faces [F,3] int32).  face_idx (nullable) = nearest face. */
int hold_mesh_sdf(hold_ctx* ctx, int B, int P, const float* points, int V, const float* verts, int verts_batched, int F,
                  const int32_t* faces, float* sdf, int32_t* face_idx, void* stream);
/* The per-ray reduction of check_off_in_surface_points_cano_mesh (volsdf_utils.py:209-217): over the S samples of each of
 * R rays, off_surface = min sdf > threshold, in_surface = min sdf <= 0 (uint8 flags, each output nullable). */
int hold_off_in_surface(hold_ctx* ctx, int R, int S, const float* sdf, float threshold, uint8_t* off_surface,
                        uint8_t* in_surface, void* stream);
/* GPU Multiresolution IsoSurface Extraction (SURVEY §8f rank 4) — the class `mise.MISE` of code/src/libmise/mise.pyx (the
 * reference's only native code) as driven by generate_mesh (utils/meshing.py:9-72): same query / update / to_dense rounds,
 * same dense (R+1)^3 value grid, R = resolution_0 << depth, bit for bit; marching cubes stays with the caller (skimage).
 *   create   : MISE.__cinit__ (mise.pyx:47-88)
 *   query    : MISE.query  -> lattice coordinates [n,3] int32 of the points without a value (device buffer `coords` of
 *              `capacity` points, may be NULL to only count); *n_points on the host (one stream sync per round)
 *   update   : MISE.update -> values [n] in the order of the last query; marks and subdivides active voxels
 *   to_dense : MISE.to_dense -> out [(R+1)^3] float32, x-major like the reference's array */
typedef struct hold_mise hold_mise;
int hold_mise_create(hold_ctx* ctx, int resolution_0, int depth, float threshold, hold_mise** out, void* stream);
int hold_mise_query(hold_mise* h, int32_t* coords, int capacity, int* n_points, void* stream);
int hold_mise_update(hold_mise* h, const float* values, int n_values, void* stream);
int hold_mise_to_dense(hold_mise* h, float* out, void* stream);

/* Marching cubes on the dense value grid vol [n0,n1,n2] (C order) — the last step of generate_mesh (utils/meshing.py:51, which calls
 * skimage.measure.marching_cubes_lewiner; skimage is absent from this image, so this is a classic case-table marching cubes whose
 * tables are DERIVED (tools/gen_mc_tables.py), pinned to oracle/marching_cubes.py bit for bit and to geometric properties, not to
 * Lewiner's triangulation).  A node is inside when value < level; one vertex per grid edge whose ends differ, at lower_end +
 * (level - v0) / (v1 - v0), index coordinates; normals (right-hand rule) towards increasing values.
 *   hold_mc_mark: edge_flags [n0*n1*n2, 3] int32 (vertex on the edge from node along axis?), cell_ntri [(n0-1)(n1-1)(n2-1)] int32.
 *   The caller forms the exclusive scans edge_vid / cell_off (int64) of both arrays; their totals size verts [Nv,3] and faces [Nt,3].
 *   hold_mc_emit: writes the vertices and the faces (vertex ids) in scan order. */
int hold_mc_mark(hold_ctx* ctx, int n0, int n1, int n2, const float* vol, float level, int32_t* edge_flags, int32_t* cell_ntri, void* stream);
int hold_mc_emit(hold_ctx* ctx, int n0, int n1, int n2, const float* vol, float level, const int32_t* edge_flags, const int64_t* edge_vid,
                 const int64_t* cell_off, float* verts, int32_t* faces, void* stream);
int hold_mise_destroy(hold_mise* h);
/* a17: ObjectModel.forward (model/obj/object_model.py:29-70). */
int hold_object_tf(hold_ctx* ctx, int B, const float* rot /*[B,3]*/, const float* trans /*[B,3]*/,
                   const float* scene_scale /*[B]*/, float obj_scale, const float* denorm_mat /*[4,4]*/,
                   const float* pts_cano /*[Nv,3]*/, int Nv, float* tfs /*[B,4,4]*/, float* verts /*[B,Nv,3] or NULL*/,
                   void* stream);
/* a1: get_camera_params (datasets/utils.py:255-282): uv [B,P,2], pose [B,4,4], K [B,4,4] ->
 * ray_dirs [B*P,3], cam_loc [B*P,3] (cam_loc repeated per ray as mano_node.py:90-92). */
int hold_camera_rays(hold_ctx* ctx, int B, int P, const float* uv, const float* pose, const float* intrinsics,
                     float* ray_dirs, float* cam_loc, void* stream);

/* a4: ErrorBoundSampler.get_z_vals (engine/ray_sampler.py:128-352) driving sdf_func_with_deformer
 * (engine/volsdf_utils.py:150-169).  R rays = B frames x R/B rays, frame-major.
 * z_vals [R, n_samples + n_samples_extra + 2]; iters: device int32 = rounds executed (batch-global). */
int hold_sample(hold_ctx* ctx, int node, int R, int B, const float* cam_loc, const float* ray_dirs,
                const hold_node_pose* pose, const hold_sampler_rand* rnd, float* z_vals, int32_t* iters,
                void* stream);

/* One iteration of the while loop of ErrorBoundSampler.get_z_vals (engine/ray_sampler.py:160-311) on caller-supplied state
 * ("teacher forcing": lets a test compare a single round with the reference without upstream last-bit noise).
 * z_old/sdf_old [R, it*N_eval] sorted state of the previous rounds (NULL for it == 0), z_new/sdf_new [R, N_eval] this round's
 * samples, beta_in/far [R].  Outputs: merged (z, sdf) [R, (it+1)*N_eval] (optional), beta_out [R] after the line search
 * (:208-220), samples_out = the next round's N_eval samples (:246-307) when the batch-global flag says upsample, else the final
 * sorted z_vals [R, N + N_extra + 2] (:313-336); *upsample_out_host (HOST int) tells which.  Synchronises the stream. */
int hold_sampler_round(hold_ctx* ctx, int node, int R, int it, const float* z_old, const float* sdf_old, const float* z_new,
                       const float* sdf_new, const float* beta_in, const float* far, const float* beta_param,
                       float* z_merged, float* sdf_merged, float* beta_out, float* samples_out, int32_t* upsample_out_host,
                       void* stream);
/* a5+a10+a11+a12: Node.forward after sampling (node.py:55-86): inverse warp, SDF + feature + gradient,
 * forward-skinning Jacobian, normals, colour net, Laplace density.  out->z_vals is an INPUT here. */
int hold_shade(hold_ctx* ctx, int node, int R, int B, int S, const float* cam_loc, const float* ray_dirs,
               const hold_node_pose* pose, const hold_factors* out, void* stream);
/* a13+a14: merge_factors + volumetric_render for the composite and for each node
 * (hold/hold_net.py:76-88).  comp_S = n*S - 2n + 1.  per_node[k] may be NULL. */
int hold_composite(hold_ctx* ctx, int n, int R, int S, const hold_factors* factors /*[n]*/,
                   const int32_t* class_ids_host /*[n]*/, const hold_render_out* comp,
                   const hold_render_out* per_node /*[n] or NULL*/, void* stream);

/* Reverse mode of hold_composite (torch.autograd through merge_factors + density2weight + the integrals of volumetric_render in
 * training, hold/hold_utils.py:76-121,243-271): upstream gradients of the composite render (g_comp) and / or of the n per-node
 * renders (g_per_node[n]) -> gradients w.r.t. every node's color [R,S,3], normal [R,S,3] and density [R,S] (d_factors[k], overwritten;
 * z_vals carry no gradient: the sampler runs under no_grad).  In a hold_render_out used as gradient any pointer may be NULL (= 0);
 * fg_weights is ignored.  mask_prob's clamp(0, 1) passes the gradient where 0 <= sum(w) <= 1. */
int hold_composite_bwd(hold_ctx* ctx, int n, int R, int S, const hold_factors* factors, const int32_t* class_ids_host,
                       const hold_render_out* g_comp, const hold_render_out* g_per_node, const hold_factors* d_factors, void* stream);
/* a18 (foreground): the whole path for n nodes, one call, no host sync. node_ids[k] are ctx node slots. */
int hold_render_fg(hold_ctx* ctx, int n, const int32_t* node_ids_host, int R, int B, const float* cam_loc,
                   const float* ray_dirs, const hold_node_pose* poses /*[n]*/, const hold_factors* factors /*[n]*/,
                   const hold_render_out* comp, const hold_render_out* per_node /*[n] or NULL*/,
                   int32_t* iters /*[n] device*/, void* stream);

/* SURVEY §8f rank 1 — the NeRF++ background (model/renderables/background.py).
 * hold_bg_set_weights: Background.bg_implicit_network (9 plain layers `lin<k>.{weight,bias}`: weight_g NULL) and
 * Background.bg_rendering_network (2 plain layers, 315 -> 128 -> 3); mlp_mode = HOLD_MLP_* arithmetic of both nets.
 * hold_background: HOLDNet.forward's background leg (hold/hold_net.py:91-118,125-134): inverse_sample +
 * Background.forward.  fg_bg_weights [R] is volumetric_render's `bg_weights`; frame_code [B,32] is
 * Background.frame_latent_encoder(idx).  Outputs (any may be NULL): bg_rgb [R,3] (= bg_weights * bg_rgb_only),
 * bg_rgb_only [R,3], bg_semantics [R,4], bg_z_vals [R,32]. */
int hold_bg_set_weights(hold_ctx* ctx, const hold_mlp_weights* sdf, const hold_mlp_weights* rgb, int mlp_mode, void* stream);
int hold_background(hold_ctx* ctx, int R, int B, const float* cam_loc, const float* ray_dirs, const float* frame_code,
                    const float* fg_bg_weights, float* bg_rgb, float* bg_rgb_only, float* bg_semantics,
                    float* bg_z_vals, void* stream);

/* Building blocks exported for tests and for callers that hold canonical points already
 * (hold_utils.query_oc, meshing): ImplicitNet.forward on canonical points (shape_net.py:84-130). */
int hold_sdf_eval(hold_ctx* ctx, int node, int P, const float* x_c /*[P,3]*/, const float* embed_w,
                  float* sdf /*[P]*/, float* grad /*[P,3] or NULL*/, float* feat /*[P,256] or NULL*/, void* stream);

/* RenderingNet.forward, mode "pose" (networks/texture_net.py:46-101): P = B x points-per-frame canonical points x_c [P,3],
 * normals [P,3], feature vectors [P,256]; hand: pose_cond [B,45] (= cond["pose"], lin_pose applied inside); object:
 * time_code [B,32] (the reference concatenates it to the features, engine/volsdf_utils.py:133-141).  -> rgb [P,3]. */
int hold_rgb_eval(hold_ctx* ctx, int node, int B, int P, const float* x_c, const float* normals, const float* pose_cond,
                  const float* feat, const float* time_code, float* rgb, void* stream);

/* ---- SURVEY §8f rank 2: building blocks of the training backward (hold/hold.py:110-137; algebra in hold_b200/train_algo.py).
 * hold_linear: C[P, nvalid] = A[P, kvalid] . M^T (+ bias) in fp32-level arithmetic (tcgen05, fp16 hi/lo split x 3 passes) against one
 * of the node's packed matrices M, selected by `mat`:
 *    0..8    SDF W_l (networks/shape_net.py:118-126; W_4 carries the skip's 1/sqrt 2, l = 8: the 256 feature rows), bias b_l
 *    16..24  SDF W_l^T (A has N_l columns, C has K_l: 39 for l = 0)
 *    32..35  colour W_l, l = 0..3 (texture_net.py:95-100); l = 0 takes A in the order [feature (256) | x_c, n, pose (14) | time code (32)]
 *    48, 49  colour W_0^T: to the 256 feature inputs / to the other inputs [x_c, n, pose (14) | time code (32)];  50..52  colour W_1..3^T
 * node = -1 addresses the background nets (model/renderables/background.py; packed by hold_bg_set_weights with HOLD_MLP_TC): 0..8 the
 * implicit net's W_l (lin0: 116 inputs = PE-10 of the 4-d point (84) + frame code (32); lin3: 172 outputs, the skip re-feeds the 84 embedding columns), 16..24 their transposes, 32 the colour
 * head's lin0 (315 -> 128, A in the order [feature (256) | view PE-4 (27), frame code (32)]), 48 / 49 its transpose to the features / to
 * [view, frame code].
 * A and C rows must be 16-byte aligned (lda, ldc multiples of 4).  in_scale: device scalar (power of two) or NULL — A is fed as
 * A / in_scale and C multiplied back, which keeps small gradients inside the split's range. */
int hold_linear(hold_ctx* ctx, int node, int mat, int P, const float* A, int lda, int kvalid, int add_bias, const float* in_scale,
                float* C, int ldc, int nvalid, void* stream);

/* Weight-gradient reduction over the points, out[n, k] = sum_p D[p, n] * A[p, k] (N, K <= 256; out [N, ldo] is overwritten), on
 * tcgen05 with the same fp16 hi/lo split x 3 passes (hold_b200/csrc/wgrad_tc.cuh).  d_scale / a_scale: device scalars (powers of
 * two, NULL = 1) by which D / A are divided before the split; the result is multiplied back. */
int hold_wgrad(hold_ctx* ctx, int P, const float* D, int ldd, int N, const float* A, int lda, int K, const float* d_scale,
               const float* a_scale, float* out, int ldo, void* stream);

/* *scale_out (device) = 2^floor(log2(max |x|)) of the [P, ncols] matrix x (1e-30 floor): the operand scale hold_linear / hold_wgrad take. */
int hold_pow2_scale(hold_ctx* ctx, int P, int ncols, const float* x, int ld, float* scale_out, void* stream);

/* Pointwise steps of the training backward on [P, ld] fp32 matrices (hold_b200/csrc/train.cuh): op 0 ACT out0 = [softplus(z) | e],
 * out1 = softplus'(z); 1 MUL; 2 MULROW (in0 = one row); 3 U_DZ2 out0 = h s, out1 = h q softplus''(z); 4 DZ out0 = in0 in1 (+ in2);
 * 5 EMBED (aux = derivative order 0..2; in1 = BARF weights or NULL); 6 EMBED_VJP; 7 EMBED_JVP; 8 RELU; 9 RELU_BWD. */
typedef struct hold_ew_args {
  const float* in0; const float* in1; const float* in2;
  float* out0; float* out1;
  int32_t ld_in0, ld_in1, ld_in2, ld_out0, ld_out1;
  int32_t ncols, aux;
} hold_ew_args;
int hold_train_ew(hold_ctx* ctx, int op, int P, const hold_ew_args* args, void* stream);
/* KNNDeformer.forward(inverse=True) / ObjectDeformer.forward(inverse=True): x [B,P,3] -> x_c, knn idx [B,P,15] (opt). */
int hold_inverse_warp(hold_ctx* ctx, int node, int B, int P, const float* x, const hold_node_pose* pose,
                      float* x_c, int32_t* knn_idx, uint8_t* outlier_mask, void* stream);

/* KNNDeformer.forward_skinning (model/mano/deformer.py:70-82) / ObjectDeformer.forward_skinning (model/obj/deformer.py:40-46):
 * canonical points x_c [B,P,3] -> deformed points x_d [B,P,3]; hand: 15 nearest CANONICAL vertices, blended transform applied
 * as is (skinning(inverse=False), deformer.py:167-170); knn_idx [B,P,15] / outlier_mask [B,P] optional (hand only). */
int hold_forward_warp(hold_ctx* ctx, int node, int B, int P, const float* x_c, const hold_node_pose* pose, float* x_d,
                      int32_t* knn_idx, uint8_t* outlier_mask, void* stream);

/* Reverse mode of hold_inverse_warp w.r.t. the transforms (skinning weights are detached in the reference, deformer.py:101):
 * g_xc [B,P,3] -> g_tfs (hand [B,16,4,4], object [B,4,4]; the constant last row gets 0 except [3][3]) and, optionally, g_x
 * [B,P,3].  Hand nodes need the forward's knn_idx [B,P,15].  With hold_sdf_eval's d sdf / d x_c upstream and
 * hold_mano_lbs_bwd (g_tfs) downstream this is a joint SDF + LBS backward for pose refinement (BASELINE configs[4]). */
int hold_inverse_warp_bwd(hold_ctx* ctx, int node, int B, int P, const float* x, const hold_node_pose* pose, const int32_t* knn_idx,
                          const float* g_xc, float* g_tfs, float* g_x, void* stream);

/* ---- Fused glue of the training forward and its reverse mode (hold_b200/csrc/train_glue.cuh; arithmetic in train_glue_phases.h).
 * Every stash, scratch and output is caller-allocated (a node's stash must survive until its backward, whatever other nodes run in
 * between); no call allocates or synchronises the host, so a training step that uses them stays capturable as one CUDA graph.
 *
 * hold_train_glue_sizes: floats of the stash hold_normal_density writes for B x P points of `node` (hand 25, object 9 per point)
 * and of the scratch hold_normal_density_bwd needs (per-block partial sums).  Either pointer may be NULL. */
int hold_train_glue_sizes(hold_ctx* ctx, int node, int B, int P, int64_t* stash_floats, int64_t* scratch_floats);
/* extract_features' normal and the Laplace density in training (engine/volsdf_utils.py:66-102, engine/density.py:21-26) for
 * frame-major points [B,P]: J = (sum_j w_j tfs_j)[:3,:3] with w the detached skinning weights of x_c's 15 nearest CANONICAL
 * vertices (hand; tfs [B,16,4,4]) or tfs[:3,:3] (object; tfs [B,4,4], x_c unused and may be NULL); g = d sdf / d x_c [B*P,3],
 * sdf [B*P], beta: device scalar, the effective beta (|beta| + beta_min).  -> normal = normalize(g . J^-1, eps 1e-6) [B*P,3],
 * density [B*P], stash (hold_train_glue_sizes) for the backward. */
int hold_normal_density(hold_ctx* ctx, int node, int B, int P, const float* x_c, const float* grad, const float* sdf,
                        const float* tfs, const float* beta, float* normal, float* density, float* stash, void* stream);
/* Reverse mode of hold_normal_density from its stash: seeds d_normal [B*P,3] and d_density [B*P] (each may be NULL = 0) ->
 * d_grad [B*P,3], d_sdf [B*P] (0 where sdf == 0), d_tfs (overwritten; only the 3x3 blocks are non-zero) and d_beta [1].  scratch:
 * hold_train_glue_sizes.  Fixed-order sums: bitwise reproducible from run to run. */
int hold_normal_density_bwd(hold_ctx* ctx, int node, int B, int P, const float* grad, const float* sdf, const float* beta,
                            const float* stash, const float* d_normal, const float* d_density, float* d_grad, float* d_sdf,
                            float* d_tfs, float* d_beta, float* scratch, void* stream);
/* The background's network inputs for R rays (background.py:35-100): for the 32 inverse-sphere depths of every ray, emb_pts
 * [R*32,84] = PE-10 of depth2pts_outside (:102-135) and emb_view [R*32,27] = PE-4 of the ray direction. */
int hold_bg_inputs(hold_ctx* ctx, int R, float r_sphere, const float* cam_loc, const float* ray_dirs, float* emb_pts,
                   float* emb_view, void* stream);
/* bg_volume_rendering of the 32 samples per ray (background.py:137-165) + Background.forward's outputs: sdf at sdf[(r*32+k)*ld_sdf]
 * (column 0 of the background SDF net's [R*32, 257] output: ld_sdf = 257), rgb [R*32,3], fg_bg_weights [R] -> bg_rgb [R,3],
 * bg_rgb_only [R,3], bg_semantics [R,4] (each may be NULL). */
int hold_bg_integrate(hold_ctx* ctx, int R, float r_sphere, const float* sdf, int ld_sdf, const float* rgb, const float* fg_bg_weights,
                      float* bg_rgb, float* bg_rgb_only, float* bg_semantics, void* stream);
/* Reverse mode of hold_bg_integrate: seeds of its three outputs (each may be NULL = 0) -> d_rgb [R*32,3], d_sdf [R*32] (contiguous;
 * 0 where sdf == 0), d_fg_bg_weights [R]. */
int hold_bg_integrate_bwd(hold_ctx* ctx, int R, float r_sphere, const float* sdf, int ld_sdf, const float* rgb,
                          const float* fg_bg_weights, const float* g_bg_rgb, const float* g_bg_rgb_only, const float* g_bg_semantics,
                          float* d_rgb, float* d_sdf, float* d_fg_bg_weights, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HOLD_B200_H */
