"""Training-mode forward/backward of a node on the GPU (SURVEY §8f rank 2; hold/hold.py:110-137, model/renderables/node.py:49-87,
engine/volsdf_utils.py:51-147 with `create_graph=is_training`).

torch.autograd.Functions whose forward AND backward run the algebra of hold_b200/train_algo.py on libhold_b200.so:
  * every product with a weight matrix: `hold_linear` — the tcgen05 split-precision GEMM (k_mlp_tc<MLP_LINEAR>) against the node's
    packed weight images (forward and transposed);
  * every pointwise step between them: `hold_train_ew` (hold_b200/csrc/train.cuh);
  * the weight-gradient reductions dW = D^T A over the points: `hold_wgrad` (k_wgrad_tc: tcgen05 with in-register transposition
    of both operands, same split-precision arithmetic);
  * inverse skinning / rigid warp and the pose servers: the existing kernels and their backward twins (hold_inverse_warp_bwd,
    hold_mano_lbs_bwd, hold_object_tf_bwd).
The second-order path of the reference (normals feed the colour net with create_graph=True) needs no double backward here:
d sdf / d x_c is an OUTPUT of SdfNetFn and its backward takes a seed for it (train_algo.sdf_backward).

What stays in PyTorch on purpose (host code per BASELINE.json north_star: "Host code stays Python/PyTorch for the training loop"):
weight-norm folding of the parameters, losses, the optimiser; and, by default, the per-point 3x3 normal algebra, the Laplace
density and the background's inputs and 32-sample integration.  fused=True (node_forward_train, background_forward_train,
forward_train, TrainStep) runs that glue on hold_normal_density / hold_bg_inputs / hold_bg_integrate and their backward twins
(NormalDensityFn, BgIntegrateFn; hold_b200/csrc/train_glue.cuh) instead."""
from __future__ import annotations

import ctypes as C
import math

import torch

from . import capi, train_algo as T
from .capi import EwArgs, NodePose, check, lib, ptr, stream_ptr

WGRAD_TC = True   # weight-gradient reductions on hold_wgrad (tcgen05); False: torch.matmul (fp32 library GEMM), kept for A/B timing

EW = dict(ACT=0, MUL=1, MULROW=2, U_DZ2=3, DZ=4, EMBED=5, EMBED_VJP=6, EMBED_JVP=7, RELU=8, RELU_BWD=9)


def fold(lin):
    """weight-norm fold of one layer of the mirror (nn.utils.weight_norm, dim=0), tracked by autograd."""
    if hasattr(lin, "weight_v"):
        return lin.weight_v * (lin.weight_g / lin.weight_v.norm(dim=1, keepdim=True))
    return lin.weight


def _ld(t):
    assert t.dim() == 2 and t.stride(1) == 1, "row-major matrix (rows may be strided)"
    return t.stride(0)


def _ew(node, op, P, ncols, in0, in1=None, in2=None, out0=None, out1=None, aux=0, ld2=None):
    a = EwArgs()
    a.in0, a.in1, a.in2 = in0.data_ptr(), (in1.data_ptr() if in1 is not None else None), (in2.data_ptr() if in2 is not None else None)
    a.out0, a.out1 = out0.data_ptr(), (out1.data_ptr() if out1 is not None else None)
    a.ld_in0 = _ld(in0) if in0.dim() == 2 else 0
    a.ld_in1 = (_ld(in1) if in1.dim() == 2 else 0) if in1 is not None else 0
    a.ld_in2 = ((_ld(in2) if in2.dim() == 2 else 0) if in2 is not None else 0) if ld2 is None else ld2
    a.ld_out0 = _ld(out0)
    a.ld_out1 = _ld(out1) if out1 is not None else 0
    a.ncols, a.aux = ncols, aux
    check(lib().hold_train_ew(node.ctx.h, op, P, C.byref(a), stream_ptr()))


class CudaOps:
    """train_algo backend on libhold_b200.so.  net = "sdf" | "rgb".  Activations live in [P,256] (or [P,320]) row buffers."""

    def __init__(self, node, net, W, b):
        self.node, self.net, self.W, self.b = node, net, W, b   # W, b: folded fp32 tensors (detached), reference column order
        self.scaled = False                                       # backward: scale operands by a power of two (hold_linear in_scale)
        self.hand = node.kind == "hand"

    # ---- products with a weight matrix
    def _linear(self, mat, A, kvalid, nvalid, bias, out_cols=256):
        P = A.shape[0]
        assert A.stride(1) == 1 and A.stride(0) % 4 == 0 and A.data_ptr() % 16 == 0, "hold_linear wants 16-byte aligned rows"
        out = torch.empty(P, out_cols, device=A.device)
        sc = self._scale(A) if self.scaled else None
        check(lib().hold_linear(self.node.ctx.h, self.node.slot, mat, P, ptr(A) if A.is_contiguous() else C.c_void_p(A.data_ptr()), A.stride(0),
                                kvalid, 1 if bias else 0, ptr(sc), C.c_void_p(out.data_ptr()), out.stride(0), nvalid, stream_ptr()))
        return out[:, :nvalid]

    def _scale(self, t):
        """device scalar 2^floor(log2 max|t|) (hold_pow2_scale: two small launches, no host sync)"""
        sc = torch.empty(1, device=t.device)
        check(lib().hold_pow2_scale(self.node.ctx.h, t.shape[0], t.shape[1], C.c_void_p(t.data_ptr()), t.stride(0), ptr(sc), stream_ptr()))
        return sc

    def lin(self, A, l, bias=True):
        if self.net == "sdf":
            if l == 8:   # [sdf head | 256 feature rows]: the head is a matrix-vector product
                feat = self._linear(8, A, 256, 256, bias)
                head = A @ self.W[8][0] + (self.b[8][0] if bias else 0.0)
                return torch.cat([head[:, None], feat], 1)
            n = T.N_SKIP_A if l == 3 else 256
            return self._linear(l, A, A.shape[1], n, bias)
        if l == 4:       # 3-row sigmoid head
            y = A @ self.W[4].T
            return y + self.b[4] if bias else y
        if l == 0:       # kernel operand order: [feature (256) | x_c, n, pose (14) | time code (32)]
            A = torch.cat([A[:, 14:270], A[:, :14], A[:, 270:], A.new_zeros(A.shape[0], 320 - A.shape[1])], 1)
            return self._linear(32, A, 320, 256, bias)
        return self._linear(32 + l, A, 256, 256, bias)

    def lin_t(self, A, l):
        if self.net == "sdf":
            if l == 8:
                d_feat = A[:, 1:].contiguous()
                return A[:, :1] * self.W[8][0][None, :] + self._linear(24, d_feat, 256, 256, False)
            if l == 0:
                return self._linear(16, A, 256, T.D_EMBED, False, out_cols=40)
            return self._linear(16 + l, A, A.shape[1], 256, False)
        if l == 4:
            return A @ self.W[4]
        if l == 0:
            k0 = self.W[0].shape[1]
            f = self._linear(48, A, 256, 256, False)
            o = self._linear(49, A, 256, 64, False, out_cols=64)
            return torch.cat([o[:, :14], f, o[:, 14:14 + (k0 - 270)]], 1)
        return self._linear(49 + l, A, 256, 256, False)

    def wgrad(self, D, A):
        """D^T A over the points: hold_wgrad (tcgen05, operands rescaled by powers of two) in blocks of <= 256 x 256."""
        if not WGRAD_TC:
            return D.T @ A
        P, N = D.shape
        K = A.shape[1]
        assert D.stride(1) == 1 and A.stride(1) == 1
        out = torch.empty(N, K, device=D.device)
        sd, sa = self._scale(D), self._scale(A)
        for n0 in range(0, N, 256):
            for k0 in range(0, K, 256):
                check(lib().hold_wgrad(self.node.ctx.h, P, C.c_void_p(D.data_ptr() + 4 * n0), D.stride(0), min(256, N - n0),
                                       C.c_void_p(A.data_ptr() + 4 * k0), A.stride(0), min(256, K - k0), ptr(sd), ptr(sa),
                                       C.c_void_p(out.data_ptr() + 4 * (n0 * K + k0)), K, stream_ptr()))
        return out

    def colsum(self, D):
        return D.sum(0)

    def w_row(self):
        return self.W[8][0]

    # ---- pointwise steps: hold_train_ew
    def act(self, z, e=None):
        P, n = z.shape
        a, s = torch.empty(P, 256, device=z.device), torch.empty(P, 256, device=z.device)
        _ew(self.node, EW["ACT"], P, n, z, e, None, a, s, aux=0 if e is None else e.shape[1])
        return (a[:, :n] if e is None else a[:, :n + e.shape[1]]), s[:, :n]

    def _binary(self, op, x, y, in2=None, ld2=None, two=False):
        P, n = y.shape
        o0 = torch.empty(P, 256 if n <= 256 else 320, device=y.device)
        o1 = torch.empty_like(o0) if two else None
        _ew(self.node, op, P, n, x, y, in2, o0, o1, ld2=ld2)
        return (o0[:, :n], o1[:, :n]) if two else o0[:, :n]

    def mul(self, x, y):
        return self._binary(EW["MUL"], x, y)

    def mulrow(self, row, y):
        return self._binary(EW["MULROW"], row.contiguous(), y)

    def u_dz2(self, h, s, q):
        if q.stride(0) == 0:   # q_7 = w broadcast over the points
            return self._binary(EW["U_DZ2"], h, s, q[0].contiguous(), ld2=0, two=True)
        return self._binary(EW["U_DZ2"], h, s, q, two=True)

    def dz(self, dA, s, dz2):
        return self._binary(EW["DZ"], dA, s, dz2)

    def embed(self, x, embed_w, order):
        P = x.shape[0]
        out = torch.empty(P, 40, device=x.device)
        xc = x.contiguous()
        _ew(self.node, EW["EMBED"], P, 40, xc, embed_w, None, out, aux=order)
        return out[:, :T.D_EMBED]

    def embed_vjp(self, d1, ge):
        P = d1.shape[0]
        out = torch.empty(P, 3, device=d1.device)
        _ew(self.node, EW["EMBED_VJP"], P, 3, d1, ge, None, out)
        return out

    def embed_jvp(self, d1, v):
        P = d1.shape[0]
        out = torch.empty(P, 40, device=d1.device)
        _ew(self.node, EW["EMBED_JVP"], P, 40, d1, v.contiguous(), None, out)
        return out[:, :T.D_EMBED]

    def relu(self, z):
        P, n = z.shape
        out = torch.empty(P, 256, device=z.device)
        _ew(self.node, EW["RELU"], P, n, z, None, None, out)
        return out[:, :n]

    def relu_bwd(self, dA, a):
        return self._binary(EW["RELU_BWD"], dA, a)


def _folded_sdf(node):
    W = [fold(getattr(node.implicit_network, f"lin{l}")) for l in range(9)]
    b = [getattr(node.implicit_network, f"lin{l}").bias for l in range(9)]
    return W, b


def _folded_rgb(node):
    W = [fold(getattr(node.rendering_network, f"lin{l}")) for l in range(5)]
    b = [getattr(node.rendering_network, f"lin{l}").bias for l in range(5)]
    return W, b


class SdfNetFn(torch.autograd.Function):
    """(sdf [P], feat [P,256], g = d sdf / d x_c [P,3]) = ImplicitNet(x_c); differentiable w.r.t. x_c and the folded weights,
    including through g (the reference's create_graph=True path)."""

    @staticmethod
    def forward(fctx, node, x, *Wb):
        fctx.set_materialize_grads(False)
        W, b = [w.detach().float() for w in Wb[:9]], [v.detach().float() for v in Wb[9:]]
        Wk = list(W)
        Wk[0] = W[0][:, :T.D_EMBED].contiguous()     # hand: the 45 pose-condition columns are multiplied by zero (shape_net.py:104-106)
        ops = CudaOps(node, "sdf", Wk, b)
        sdf, feat, g, st = T.sdf_forward(ops, x.detach().float().contiguous(), node.embed_w())
        fctx.ops, fctx.st, fctx.k0 = ops, st, W[0].shape[1]
        return sdf.contiguous(), feat.contiguous(), g

    @staticmethod
    def backward(fctx, d_sdf, d_feat, d_g):
        ops = fctx.ops
        ops.scaled = True
        f = lambda t: None if t is None else t.float().contiguous()
        d_x, dW, db = T.sdf_backward(ops, fctx.st, f(d_sdf), f(d_feat), f(d_g))
        dW[4] = dW[4] * (1.0 / math.sqrt(2.0))       # the packed W_4 carries the skip's 1/sqrt 2
        if fctx.k0 > T.D_EMBED:
            dW[0] = torch.cat([dW[0], dW[0].new_zeros(256, fctx.k0 - T.D_EMBED)], 1)
        return (None, d_x, *dW, *db)


class RgbNetFn(torch.autograd.Function):
    """rgb [P,3] = RenderingNet([x_c, n, pose_embed, feat (, time)]) (texture_net.py:69-101); differentiable w.r.t. the input
    matrix and the folded weights."""

    @staticmethod
    def forward(fctx, node, inp, *Wb):
        W, b = [w.detach().float() for w in Wb[:5]], [v.detach().float() for v in Wb[5:]]
        ops = CudaOps(node, "rgb", W, b)
        rgb, st = T.rgb_forward(ops, inp.detach().float().contiguous())
        fctx.ops, fctx.st = ops, st
        return rgb

    @staticmethod
    def backward(fctx, d_rgb):
        fctx.ops.scaled = True
        d_in, dW, db = T.rgb_backward(fctx.ops, fctx.st, d_rgb.float().contiguous())
        return (None, d_in, *dW, *db)


class InverseWarpFn(torch.autograd.Function):
    """x_c = deformer.forward(x, tfs, inverse=True) (mano/deformer.py:34-68,145-170; obj/deformer.py:10-31); differentiable w.r.t.
    tfs (skinning weights are detached in the reference, deformer.py:101) and x."""

    @staticmethod
    def forward(fctx, node, x, tfs, verts):
        B, P, _ = x.shape
        dev = x.device
        pose = NodePose()
        tf = tfs.detach().float().contiguous()
        pose.tfs = tf.data_ptr()
        keep = [tf]
        hand = node.kind == "hand"
        if hand:
            vv = verts.detach().float().contiguous()
            pose.posed_verts = vv.data_ptr()
            keep.append(vv)
        xi = x.detach().float().contiguous()
        xc = torch.empty(B, P, 3, device=dev)
        idx = torch.empty(B, P, 15, dtype=torch.int32, device=dev) if hand else None
        check(lib().hold_inverse_warp(node.ctx.h, node.slot, B, P, ptr(xi), C.byref(pose), ptr(xc), ptr(idx), None, stream_ptr()))
        fctx.node, fctx.keep, fctx.idx, fctx.xi, fctx.hand = node, keep, idx, xi, hand
        return xc

    @staticmethod
    def backward(fctx, g_xc):
        node, xi = fctx.node, fctx.xi
        B, P, _ = xi.shape
        pose = NodePose()
        pose.tfs = fctx.keep[0].data_ptr()
        if fctx.hand:
            pose.posed_verts = fctx.keep[1].data_ptr()
        g = g_xc.float().contiguous()
        g_tfs = torch.zeros_like(fctx.keep[0])
        g_x = torch.empty_like(xi)
        check(lib().hold_inverse_warp_bwd(node.ctx.h, node.slot, B, P, ptr(xi), C.byref(pose), ptr(fctx.idx), ptr(g), ptr(g_tfs), ptr(g_x), stream_ptr()))
        return None, g_x, g_tfs, None


def laplace_density(sdf, beta):
    """engine/density.py:21-26."""
    return (1.0 / beta) * (0.5 + 0.5 * sdf.sign() * torch.expm1(-sdf.abs() / beta))


def _glue_sizes(node, B, P):
    """floats of hold_normal_density's stash and of hold_normal_density_bwd's scratch for B x P points of the node"""
    st, sc = C.c_int64(), C.c_int64()
    check(lib().hold_train_glue_sizes(node.ctx.h, node.slot, B, P, C.byref(st), C.byref(sc)))
    return st.value, sc.value


class NormalDensityFn(torch.autograd.Function):
    """(normal [B*P,3], density [B*P]) of a node's frame-major samples in one kernel (hold_normal_density): the normal of
    extract_features (volsdf_utils.py:66-102) = normalize(g . J^-1) with J the forward-skinning Jacobian under detached weights, and
    the Laplace density (density.py:21-26) at the effective beta.  Differentiable w.r.t. g, sdf, tfs and beta; x_c only selects
    the hand's skinning weights (detached in the reference, deformer.py:101).  The backward (hold_normal_density_bwd) reads the
    forward's per-point stash (J^-1 and the blended weights), so the KNN runs once."""

    @staticmethod
    def forward(fctx, node, B, x_c, g, sdf, tfs, beta):
        fctx.set_materialize_grads(False)
        P = x_c.shape[0] // B
        dev = g.device
        f = lambda t: t.detach().float().contiguous()
        xc, gg, s, tf, bt = f(x_c), f(g), f(sdf), f(tfs), f(beta).reshape(1)
        n_stash, _ = _glue_sizes(node, B, P)
        normal, density = torch.empty(B * P, 3, device=dev), torch.empty(B * P, device=dev)
        stash = torch.empty(n_stash, device=dev)
        check(lib().hold_normal_density(node.ctx.h, node.slot, B, P, ptr(xc), ptr(gg), ptr(s), ptr(tf), ptr(bt), ptr(normal),
                                        ptr(density), ptr(stash), stream_ptr()))
        fctx.node, fctx.B, fctx.P, fctx.keep = node, B, P, (gg, s, bt, stash)
        fctx.tfs_shape, fctx.beta_shape = tfs.shape, beta.shape
        return normal, density

    @staticmethod
    def backward(fctx, d_normal, d_density):
        node, B, P = fctx.node, fctx.B, fctx.P
        gg, s, bt, stash = fctx.keep
        dev = gg.device
        f = lambda t: None if t is None else t.float().contiguous()
        dn, dd = f(d_normal), f(d_density)
        _, n_scratch = _glue_sizes(node, B, P)
        d_g, d_s = torch.empty_like(gg), torch.empty_like(s)
        d_tfs, d_beta = torch.empty(fctx.tfs_shape, device=dev), torch.empty(1, device=dev)
        scratch = torch.empty(n_scratch, device=dev)
        check(lib().hold_normal_density_bwd(node.ctx.h, node.slot, B, P, ptr(gg), ptr(s), ptr(bt), ptr(stash), ptr(dn), ptr(dd),
                                            ptr(d_g), ptr(d_s), ptr(d_tfs), ptr(d_beta), ptr(scratch), stream_ptr()))
        return None, None, None, d_g, d_s, d_tfs, d_beta.reshape(fctx.beta_shape)


def node_forward_train(node, x, tfs, verts, frame_of_point, pose_cond=None, time_code=None, sync=True, fused=False):
    """Node.forward after sampling, training mode (node.py:57-87 + volsdf_utils.py:51-147): deformed points x [B,P,3] ->
    dict(sdf, x_c, feat, grad, normal, color, density), everything differentiable w.r.t. the node's parameters, tfs, beta,
    the frame / pose codes.  `verts`: posed vertices (hand).  frame_of_point [B*P] long.
    fused: normal and density from one kernel and its backward twin (NormalDensityFn) instead of the torch ops below."""
    if sync:
        node.sync_weights()
    B, P, _ = x.shape
    x_c = InverseWarpFn.apply(node, x, tfs, verts).reshape(B * P, 3)
    Ws, bs = _folded_sdf(node)
    sdf, feat, g = SdfNetFn.apply(node, x_c, *Ws, *bs)
    if fused:
        normal, density = NormalDensityFn.apply(node, B, x_c, g, sdf, tfs, node.density.get_beta())
    # J of forward skinning with detached weights (volsdf_utils.py:66-81): sum_j w_j tfs_j[:3,:3]; hand: KNN vs canonical verts
    elif node.kind == "hand":
        pose = NodePose()
        tf = tfs.detach().float().contiguous()
        pose.tfs = tf.data_ptr()
        idx = torch.empty(B, P, 15, dtype=torch.int32, device=x.device)
        xd = torch.empty(B, P, 3, device=x.device)
        check(lib().hold_forward_warp(node.ctx.h, node.slot, B, P, ptr(x_c.detach().reshape(B, P, 3).contiguous()), C.byref(pose), ptr(xd),
                                      ptr(idx), None, stream_ptr()))
        cano = node.server.verts_c[0]
        d2 = ((x_c.detach().reshape(B * P, 1, 3) - cano[idx.reshape(B * P, 15).long()]) ** 2).sum(-1).clamp(max=4.0)
        conf = torch.softmax(-d2, dim=1)
        w = (node.server.m["lbs_weights"][idx.reshape(B * P, 15).long()] * conf[..., None]).sum(1)         # [BP,16], detached by construction
        # points are frame-major (B blocks of P): one batched [P,16] x [16,9] product per frame instead of a per-point gather of
        # the 16 bone transforms (whose backward is a slow scatter-add)
        J = torch.bmm(w.reshape(B, P, 16), tfs[:, :, :3, :3].reshape(B, 16, 9)).reshape(B * P, 3, 3)
    else:
        J = tfs.reshape(B, 1, 4, 4)[:, :, :3, :3].expand(B, P, 3, 3).reshape(B * P, 3, 3)
    if not fused:
        # inv_ex: torch.linalg.inv reads its error flag on the host (a sync per node per step)
        normal = torch.nn.functional.normalize(torch.einsum("bi,bij->bj", g, torch.linalg.inv_ex(J).inverse), dim=1, eps=1e-6)
    if node.kind == "hand":
        pe = node.rendering_network.lin_pose(pose_cond)[:, None, :].expand(B, P, 8).reshape(B * P, 8)   # per-frame rows, frame-major points
        inp = torch.cat([x_c, normal, pe, feat], 1)
    else:
        inp = torch.cat([x_c, normal, x_c.new_zeros(B * P, 8), feat, time_code[:, None, :].expand(B, P, 32).reshape(B * P, 32)], 1)
    Wr, br = _folded_rgb(node)
    color = RgbNetFn.apply(node, inp, *Wr, *br)
    if not fused:
        density = laplace_density(sdf, node.density.get_beta())
    return dict(sdf=sdf, x_c=x_c, feat=feat, grad=g, normal=normal, color=color, density=density)


# ------------------------------------------------------------------------------------------------ scene level (hold_net.py:53-108)
def density2weight(density, z_vals, z_max):
    """engine/volsdf_utils.py:220-251."""
    dists = torch.cat([z_vals[:, 1:] - z_vals[:, :-1], z_max[:, None] - z_vals[:, -1:]], -1)
    fe = dists * density
    alpha = 1 - torch.exp(-fe)
    T = torch.exp(-torch.cumsum(torch.cat([torch.zeros_like(fe[:, :1]), fe], -1), -1))
    return alpha * T[:, :-1], T[:, -1]


def volumetric_render(f):
    """hold/hold_utils.py:243-271 (training: no fg_rgb.vis)."""
    w, bg = density2weight(f["density"], f["z_vals"], f["z_max"])
    integ = lambda v: (v * w[:, :, None]).sum(1)
    return dict(fg_rgb=integ(f["color"]), fg_weights=w, mask_prob=w.sum(1, keepdim=True).clamp(0, 1), normal=integ(f["normal"]),
                depth=integ(f["z_vals"][:, :, None]), fg_semantics=integ(f["semantics"]), bg_weights=bg)


def merge_factors(fl):
    """hold/hold_utils.py:76-121: concat on the sample axis, sort by z (stable: lower node first on ties, as the kernels do),
    drop (n-1) head / n tail entries (the reference's own asymmetry, :115-118), z_max = z_sorted[:, -n]."""
    n = len(fl)
    z = torch.cat([f["z_vals"] for f in fl], 1)
    zs, idx = torch.sort(z, dim=1, stable=True)
    out = {}
    for k in ("color", "normal", "semantics"):
        v = torch.cat([f[k] for f in fl], 1)
        out[k] = torch.gather(v, 1, idx[:, :, None].expand(-1, -1, v.shape[2]))[:, n - 1: -n]
    out["density"] = torch.gather(torch.cat([f["density"] for f in fl], 1), 1, idx)[:, n - 1: -n]
    out["z_vals"] = zs[:, n - 1: -n]
    out["z_max"] = zs[:, -n]
    return out


# ------------------------------------------------------------------------------------------------ background (renderables/background.py)
class _BgHandle:
    """What CudaOps needs from a "node" when the matrices are the background's (hold_linear with node = -1)."""

    def __init__(self, ctx):
        self.ctx, self.slot, self.kind = ctx, -1, "background"


class BgOps(CudaOps):
    """train_algo backend for the background nets: net = "bg_sdf" (9 plain layers, 116 inputs, skip at 4) | "bg_rgb" (315 -> 128 -> 3)."""

    def __init__(self, ctx, net, W, b):
        super().__init__(_BgHandle(ctx), net, W, b)

    def lin(self, A, l, bias=True):
        if self.net == "bg_sdf":
            if l == 8:
                feat = self._linear(8, A, 256, 256, bias)
                head = A @ self.W[8][0] + (self.b[8][0] if bias else 0.0)
                return torch.cat([head[:, None], feat], 1)
            return self._linear(l, A, A.shape[1], 172 if l == 3 else 256, bias)
        if l == 1:       # 128 -> 3 head
            y = A @ self.W[1].T
            return y + self.b[1] if bias else y
        A = torch.cat([A[:, 59:], A[:, :59], A.new_zeros(A.shape[0], 5)], 1)      # operand order [feature (256) | view, frame (59)] + pad
        return self._linear(32, A, 320, 128, bias)

    def lin_t(self, A, l):
        if self.net == "bg_sdf":
            if l == 8:
                return A[:, :1] * self.W[8][0][None, :] + self._linear(24, A[:, 1:].contiguous(), 256, 256, False)
            if l == 0:
                return self._linear(16, A, 256, 116, False, out_cols=116)
            return self._linear(16 + l, A, A.shape[1], 256, False)
        if l == 1:
            return A @ self.W[1]
        f = self._linear(48, A, 128, 256, False)
        o = self._linear(49, A, 128, 64, False, out_cols=64)
        return torch.cat([o[:, :59], f], 1)


class BgSdfFn(torch.autograd.Function):
    """out [P,257] = bg_implicit_network([PE-10(point) | frame code]); differentiable w.r.t. the input rows (frame code) and weights."""

    @staticmethod
    def forward(fctx, ctx, inp, *Wb):
        W, b = [w.detach().float() for w in Wb[:9]], [v.detach().float() for v in Wb[9:]]
        ops = BgOps(ctx, "bg_sdf", W, b)
        out, st = T.skipnet_forward(ops, inp.detach().float().contiguous(), skip=4, d_skip=84)
        fctx.ops, fctx.st = ops, st
        return out

    @staticmethod
    def backward(fctx, d_out):
        fctx.ops.scaled = True
        d_inp, dW, db = T.skipnet_backward(fctx.ops, fctx.st, d_out.float().contiguous())
        dW[4] = dW[4] * (1.0 / math.sqrt(2.0))
        return (None, d_inp, *dW, *db)


class BgRgbFn(torch.autograd.Function):
    """rgb [P,3] = bg_rendering_network([view PE-4 | frame code | feature]) (texture_net.py:55-68,95-101)."""

    @staticmethod
    def forward(fctx, ctx, inp, W0, W1, b0, b1):
        ops = BgOps(ctx, "bg_rgb", [W0.detach().float(), W1.detach().float()], [b0.detach().float(), b1.detach().float()])
        rgb, st = T.head_forward(ops, inp.detach().float().contiguous())
        fctx.ops, fctx.st = ops, st
        return rgb

    @staticmethod
    def backward(fctx, d_rgb):
        fctx.ops.scaled = True
        d_in, dW, db = T.head_backward(fctx.ops, fctx.st, d_rgb.float().contiguous())
        return (None, d_in, dW[0], dW[1], db[0], db[1])


def _embed_n(x, n_freq):
    out = [x]
    for k in range(n_freq):
        f = float(2.0 ** k)
        out += [torch.sin(x * f), torch.cos(x * f)]
    return torch.cat(out, -1)


def depth2pts_outside(ray_o, ray_d, depth, R_s):
    """Background.depth2pts_outside (background.py:102-135), torch (no parameters reach it)."""
    o_dot_d = (ray_d * ray_o).sum(-1)
    under = o_dot_d ** 2 - ((ray_o ** 2).sum(-1) - R_s ** 2)
    d_sphere = torch.sqrt(under) - o_dot_d
    p_sphere = ray_o + d_sphere[..., None] * ray_d
    p_mid = ray_o - o_dot_d[..., None] * ray_d
    pmn = torch.norm(p_mid, dim=-1)
    axis = torch.cross(ray_o, p_sphere, dim=-1)
    axis = axis / torch.norm(axis, dim=-1, keepdim=True)
    ang = (torch.asin(pmn / R_s) - torch.asin(pmn * depth))[..., None]
    pn = p_sphere * torch.cos(ang) + torch.cross(axis, p_sphere, dim=-1) * torch.sin(ang) + axis * (axis * p_sphere).sum(-1, keepdim=True) * (1.0 - torch.cos(ang))
    pn = pn / torch.norm(pn, dim=-1, keepdim=True)
    return torch.cat([pn, depth[..., None]], -1)


class BgIntegrateFn(torch.autograd.Function):
    """(bg_rgb [R,3], bg_rgb_only [R,3], bg_semantics [R,4]) = bg_volume_rendering of the 32 inverse-sphere samples per ray
    (background.py:137-165, AbsDensity) + Background.forward's outputs (:35-54), on hold_bg_integrate / hold_bg_integrate_bwd.
    sdf [R*32] may be a strided column (column 0 of BgSdfFn's output): the kernels take its stride, no copy.  Differentiable
    w.r.t. sdf, rgb [R*32,3] and the foreground's bg_weights [R]."""

    @staticmethod
    def forward(fctx, ctx, R_s, sdf, rgb, fg_bg_weights):
        fctx.set_materialize_grads(False)
        assert sdf.dim() == 1 and sdf.dtype == torch.float32
        R = fg_bg_weights.shape[0]
        dev = rgb.device
        s, c, w = sdf.detach(), rgb.detach().float().contiguous(), fg_bg_weights.detach().float().contiguous()
        bg_rgb, only, sem = torch.empty(R, 3, device=dev), torch.empty(R, 3, device=dev), torch.empty(R, 4, device=dev)
        check(lib().hold_bg_integrate(ctx.h, R, float(R_s), C.c_void_p(s.data_ptr()), s.stride(0), ptr(c), ptr(w), ptr(bg_rgb), ptr(only),
                                      ptr(sem), stream_ptr()))
        fctx.ctx, fctx.R_s, fctx.keep = ctx, float(R_s), (s, c, w)
        return bg_rgb, only, sem

    @staticmethod
    def backward(fctx, g_rgb, g_only, g_sem):
        s, c, w = fctx.keep
        R = w.shape[0]
        f = lambda t: None if t is None else t.float().contiguous()
        d_rgb, d_sdf, d_w = torch.empty_like(c), torch.empty(s.shape[0], device=c.device), torch.empty_like(w)
        check(lib().hold_bg_integrate_bwd(fctx.ctx.h, R, fctx.R_s, C.c_void_p(s.data_ptr()), s.stride(0), ptr(c), ptr(w), ptr(f(g_rgb)),
                                          ptr(f(g_only)), ptr(f(g_sem)), ptr(d_rgb), ptr(d_sdf), ptr(d_w), stream_ptr()))
        return None, None, d_sdf, d_rgb, d_w


def bg_inputs(ctx, ray_dirs, cam_loc, R_s):
    """The background nets' per-sample inputs without gradient (no parameter reaches them), one kernel (hold_bg_inputs):
    -> PE-10 of depth2pts_outside at the 32 inverse-sphere depths [R*32, 84], PE-4 of the ray directions [R*32, 27]."""
    R = ray_dirs.shape[0]
    dev = ray_dirs.device
    emb_pts, emb_view = torch.empty(R * 32, 84, device=dev), torch.empty(R * 32, 27, device=dev)
    check(lib().hold_bg_inputs(ctx.h, R, float(R_s), ptr(cam_loc.detach().float().contiguous()), ptr(ray_dirs.detach().float().contiguous()),
                               ptr(emb_pts), ptr(emb_view), stream_ptr()))
    return emb_pts, emb_view


def background_forward_train(bg, fg_bg_weights, ray_dirs, cam_loc, idx, B, R_s, n_bg=32, sync=True, fused=False):
    """Background.forward in training (background.py:35-100): -> dict(bg_rgb = bg_weights * bg_rgb_only, bg_rgb_only, bg_semantics),
    differentiable w.r.t. the background nets, its frame codes and the foreground's bg_weights.  Eval-mode (deterministic) inverse
    sphere samples; the nets run on hold_linear (node -1), their weights must have been packed in tensor-core mode.
    fused: the nets' inputs from one kernel (bg_inputs) and the 32-sample integration with its backward twin (BgIntegrateFn)
    instead of the torch ops below."""
    if sync:
        bg.sync_weights()
    R = ray_dirs.shape[0]
    dev = ray_dirs.device
    fc = bg.frame_latent_encoder(idx)                                                                                  # [B,32]
    fcp = fc[:, None, :].expand(B, (R // B) * n_bg, 32).reshape(R * n_bg, 32)
    Ws = [getattr(bg.bg_implicit_network, f"lin{l}").weight for l in range(9)]
    bs = [getattr(bg.bg_implicit_network, f"lin{l}").bias for l in range(9)]
    rn = bg.bg_rendering_network
    if fused:
        assert n_bg == 32, "the fused background kernels take the reference's 32 samples"
        emb_pts, view = bg_inputs(bg.ctx, ray_dirs, cam_loc, R_s)
        out = BgSdfFn.apply(bg.ctx, torch.cat([emb_pts, fcp], 1), *Ws, *bs)
        sdf, feat = out[:, 0], out[:, 1:]
        rgb = BgRgbFn.apply(bg.ctx, torch.cat([view, fcp, feat], 1), rn.lin0.weight, rn.lin1.weight, rn.lin0.bias, rn.lin1.bias)
        bg_rgb, only, sem = BgIntegrateFn.apply(bg.ctx, R_s, sdf, rgb, fg_bg_weights)
        return dict(bg_rgb=bg_rgb, bg_rgb_only=only, bg_semantics=sem)
    z = torch.flip(torch.linspace(0.0, 1.0, n_bg, device=dev) * (1.0 / R_s), dims=[-1])[None].expand(R, n_bg)       # 1/R_s ... 0
    pts = depth2pts_outside(cam_loc[:, None, :].expand(R, n_bg, 3), ray_dirs[:, None, :].expand(R, n_bg, 3), z, R_s).reshape(R * n_bg, 4)
    inp = torch.cat([_embed_n(pts, 10), fcp], 1)
    out = BgSdfFn.apply(bg.ctx, inp, *Ws, *bs)
    sdf, feat = out[:, 0], out[:, 1:]
    view = _embed_n(ray_dirs[:, None, :].expand(R, n_bg, 3).reshape(R * n_bg, 3), 4)
    rgb = BgRgbFn.apply(bg.ctx, torch.cat([view, fcp, feat], 1), rn.lin0.weight, rn.lin1.weight, rn.lin0.bias, rn.lin1.bias).reshape(R, n_bg, 3)
    dens = sdf.abs().reshape(R, n_bg)                                                                                  # AbsDensity (density.py:33-35)
    dists = torch.cat([z[:, :-1] - z[:, 1:], torch.full((R, 1), 1e10, device=dev)], -1)
    fe = dists * dens
    w = (1 - torch.exp(-fe)) * torch.exp(-torch.cumsum(torch.cat([torch.zeros(R, 1, device=dev), fe[:, :-1]], -1), -1))
    only = (w[:, :, None] * rgb).sum(1)
    sem = torch.zeros(R, 4, device=dev)
    sem[:, 0] = 1.0
    return dict(bg_rgb=fg_bg_weights[:, None] * only, bg_rgb_only=only, bg_semantics=fg_bg_weights[:, None] * sem)


class CompositeFn(torch.autograd.Function):
    """merge_factors + volumetric_render of the scene (hold_net.py:76-88) on hold_composite / hold_composite_bwd.
    inputs: per node color [R,S,3], normal [R,S,3], density [R,S] (differentiable), z_vals [R,S]; class ids.
    -> fg_rgb [R,3], mask_prob [R], normal [R,3], depth [R], fg_semantics [R,4], bg_weights [R]."""

    @staticmethod
    def forward(fctx, ctx_h, class_ids, n, *tensors):
        from .capi import Factors, RenderOut

        cols, nrms, dens, zs = tensors[:n], tensors[n:2 * n], tensors[2 * n:3 * n], tensors[3 * n:4 * n]
        R, S = zs[0].shape
        dev = zs[0].device
        f = lambda t: t.detach().float().contiguous()
        keep = [[f(cols[k]), f(nrms[k]), f(dens[k]), f(zs[k])] for k in range(n)]
        facs = (Factors * n)()
        for k in range(n):
            facs[k].color, facs[k].normal, facs[k].density, facs[k].z_vals = (t.data_ptr() for t in keep[k])
        out = dict(fg_rgb=torch.empty(R, 3, device=dev), mask_prob=torch.empty(R, device=dev), normal=torch.empty(R, 3, device=dev),
                   depth=torch.empty(R, device=dev), fg_semantics=torch.empty(R, 4, device=dev), bg_weights=torch.empty(R, device=dev))
        ro = RenderOut()
        for kk, v in out.items():
            setattr(ro, kk, v.data_ptr())
        cls = (C.c_int32 * n)(*class_ids)
        check(lib().hold_composite(ctx_h, n, R, S, facs, cls, C.byref(ro), None, stream_ptr()))
        fctx.ctx_h, fctx.cls, fctx.n, fctx.keep, fctx.facs = ctx_h, cls, n, keep, facs
        return tuple(out[k] for k in ("fg_rgb", "mask_prob", "normal", "depth", "fg_semantics", "bg_weights"))

    @staticmethod
    def backward(fctx, *gs):
        from .capi import Factors, RenderOut

        n, keep = fctx.n, fctx.keep
        R, S = keep[0][3].shape
        dev = keep[0][3].device
        g = RenderOut()
        hold = []
        for name, t in zip(("fg_rgb", "mask_prob", "normal", "depth", "fg_semantics", "bg_weights"), gs):
            if t is not None:
                t = t.float().contiguous()
                hold.append(t)
                setattr(g, name, t.data_ptr())
        d = [[torch.empty(R, S, 3, device=dev), torch.empty(R, S, 3, device=dev), torch.empty(R, S, device=dev)] for _ in range(n)]
        dfac = (Factors * n)()
        for k in range(n):
            dfac[k].color, dfac[k].normal, dfac[k].density = (t.data_ptr() for t in d[k])
        check(lib().hold_composite_bwd(fctx.ctx_h, n, R, S, fctx.facs, fctx.cls, C.byref(g), None, dfac, stream_ptr()))
        return (None, None, None, *[d[k][0] for k in range(n)], *[d[k][1] for k in range(n)], *[d[k][2] for k in range(n)], *([None] * n))


def composite(ctx, factors, class_ids):
    """dict(fg_rgb, mask_prob, normal, depth, fg_semantics, bg_weights) of the scene's factors (list of dicts with color, normal,
    density, z_vals), differentiable w.r.t. color / normal / density."""
    n = len(factors)
    fctx_set = lambda fn: fn
    outs = CompositeFn.apply(ctx.h, list(class_ids), n, *[f["color"] for f in factors], *[f["normal"] for f in factors],
                             *[f["density"] for f in factors], *[f["z_vals"] for f in factors])
    return dict(zip(("fg_rgb", "mask_prob", "normal", "depth", "fg_semantics", "bg_weights"), outs))


# ------------------------------------------------------------------------------------------------ training-mode forward (hold_net.py:53-134)
SEGM_IDS = {"bg": 0, "object": 50, "right": 150, "left": 250}     # utils/const.py:1


class PointInSpace:
    """hold/hold_utils.py:22-56: one point near each centre + a share of uniform samples in a box."""

    def __init__(self, global_sigma=0.5, global_sigma_xyz=None, local_sigma=0.01):
        self.global_sigma_xyz = torch.ones(3) * global_sigma if global_sigma_xyz is None else torch.as_tensor(global_sigma_xyz, dtype=torch.float32)
        self.local_sigma = local_sigma

    def get_points(self, pc_input, local_sigma=None, global_ratio=0.125, generator=None):
        B, N, D = pc_input.shape
        dev = pc_input.device
        sig = self.global_sigma_xyz.to(dev)
        ls = self.local_sigma if local_sigma is None else local_sigma
        local = pc_input + torch.randn(pc_input.shape, device=dev, generator=generator) * ls
        glob = torch.rand(B, int(N * global_ratio), D, device=dev, generator=generator) * (sig * 2) - sig
        return torch.cat([local, glob], 1)


pt_in_space_sampler_h = PointInSpace(global_sigma_xyz=[0.15, 0.06, 0.12])     # hold_utils.py:58


def sample_on_barycentric_mesh(verts, faces, num_samples, generator=None):
    """hold/hold_utils.py:272-304."""
    B = verts.shape[0]
    dev = verts.device
    fi = torch.randint(0, faces.shape[0], (B, num_samples), device=dev, generator=generator)
    sf = faces.long()[fi]
    v0, v1, v2 = (torch.gather(verts, 1, sf[..., k].unsqueeze(-1).expand(-1, -1, 3)) for k in range(3))
    u, v = torch.rand(B, num_samples, 1, device=dev, generator=generator), torch.rand(B, num_samples, 1, device=dev, generator=generator)
    m = u + v > 1
    u, v = torch.where(m, 1 - u, u), torch.where(m, 1 - v, v)
    return u * v0 + v * v1 + (1 - u - v) * v2


def compute_gradient_samples(sampler, node, num_pixels, verts_c, B, local_sigma=0.008, global_ratio=0.20, generator=None):
    """engine/volsdf_utils.py:19-48: grad_theta = d sdf / d x at samples around the canonical vertices (local branch) or uniform in
    [-0.3, 0.3]^3 (verts_c None); differentiable w.r.t. the SDF net (the second-order path of SdfNetFn)."""
    dev = node.density.beta.device
    if verts_c is not None:
        idx = torch.randperm(verts_c.shape[1], device=dev, generator=generator)[:num_pixels]
        sample = sampler.get_points(verts_c.index_select(1, idx), local_sigma=local_sigma, global_ratio=global_ratio, generator=generator)
    else:
        sample = torch.rand(B, num_pixels, 3, device=dev, generator=generator) * 0.6 - 0.3
    Ws, bs = _folded_sdf(node)
    _, _, g = SdfNetFn.apply(node, sample.reshape(-1, 3).contiguous(), *Ws, *bs)
    return g.reshape(sample.shape)


def prepare_loss_targets(out, node, B, P, canonical_pts, generator=None):
    """prepare_loss_targets_hand / _object (hold/hold_utils.py:149-241): <node>.index_off_surface, <node>.grad_theta and, for hands,
    <node>.pts2mano_sdf_cano / <node>.pred_sdf.  The canonical meshes are attributes the caller sets, as the reference does
    (mano_node.py:112-134 `mesh_v_cano_div`, `mesh_f_cano_div`; object_node.py:112-132 `mesh_vo_cano`, `mesh_fo_cano`); without them the
    reference skips the node's targets, and so does this."""
    from . import ops

    nid, ctx = node.node_id, node.ctx
    Ws, bs = _folded_sdf(node)
    if node.kind == "hand":
        if getattr(node, "mesh_v_cano_div", None) is None:
            return
        v = node.mesh_v_cano_div[None].repeat(B, 1, 1).float().contiguous()
        f = node.mesh_f_cano_div
        samples = pt_in_space_sampler_h.get_points(sample_on_barycentric_mesh(v, f, 256, generator), local_sigma=0.008, global_ratio=0.20, generator=generator)
        with torch.no_grad():
            out[f"{nid}.pts2mano_sdf_cano"] = ops.compute_mano_cano_sdf(ctx, v, f, samples.contiguous())
            off, _ = ops.check_off_in_surface_points_cano_mesh(ctx, v, f, canonical_pts.detach().reshape(B, -1, 3).contiguous(), B * P, threshold=0.01)
        sdf, _, _ = SdfNetFn.apply(node, samples.reshape(-1, 3).contiguous(), *Ws, *bs)            # query_oc (hold_utils.py:61-65)
        out[f"{nid}.pred_sdf"] = sdf.reshape(B, -1)
        out[f"{nid}.index_off_surface"] = off
        verts_c = node.server.verts_c.expand(B, -1, -1)
        out[f"{nid}.grad_theta"] = compute_gradient_samples(pt_in_space_sampler_h, node, 256, verts_c, B, 0.008, 0.20, generator)
    else:
        if getattr(node, "mesh_vo_cano", None) is None:
            return
        v = node.mesh_vo_cano.reshape(1, -1, 3).repeat(B, 1, 1).float().contiguous()
        with torch.no_grad():
            off, _ = ops.check_off_in_surface_points_cano_mesh(ctx, v, node.mesh_fo_cano, canonical_pts.detach().reshape(B, -1, 3).contiguous(), B * P, threshold=0.05)
        out[f"{nid}.index_off_surface"] = off
        xyz = v[0].abs().max(0).values * 1.1
        out[f"{nid}.grad_theta"] = compute_gradient_samples(PointInSpace(global_sigma_xyz=xyz.cpu()), node, 256, v, B, 0.03, 0.20, generator)


def forward_train(net, input, generator=None, fused=False):
    """HOLDNet.forward in training mode (hold/hold_net.py:53-134) -> the reference's output dict: epoch, step, fg_rgb, fg_weights-free
    composite keys (mask_prob, normal, depth, fg_semantics, bg_weights), <node>.* of every node's own volumetric_render, the loss
    targets of prepare_loss_targets, bg_z_vals, ray_dirs, cam_loc, index, and (forward) rgb, semantics, bg_rgb_only.
    Every floating-point output carries the autograd graph to the nets, beta, poses / transforms and codes.  Training-mode rules
    mirrored: pose conditioning is zeroed while current_epoch < 20 (mano_node.py:82-85); sampling runs without gradients
    (ray_sampler.py, torch.no_grad).  fused: the per-point glue of the nodes and of the background on the fused kernels
    (NormalDensityFn, bg_inputs, BgIntegrateFn)."""
    from . import ops
    from .model import ErrorBoundSampler

    uv = input["uv"]
    B, P, _ = uv.shape
    dev = uv.device
    out = {}
    if "current_epoch" in input:
        out["epoch"], out["step"] = input["current_epoch"], input.get("global_step", 0)
    early = int(input.get("current_epoch", 1 << 30)) < 20
    dirs, cam = ops.camera_rays(net.ctx, uv, input["extrinsics"], input["intrinsics"])
    fr = torch.arange(B, device=dev).repeat_interleave(P)
    factors = []
    for node in net.nodes.values():
        node.sync_weights()
        pose, keep, srv, tfs = node.articulate(input)     # servers under autograd when the pose rows require grad
        with torch.no_grad():
            z, _ = ErrorBoundSampler(node).get_z_vals(dirs, cam, pose, B)
        S = z.shape[1]
        x = (cam[:, None, :] + z[:, :, None] * dirs[:, None, :]).reshape(B, P * S, 3)
        hand = node.kind == "hand"
        pc = None
        if hand:
            pc = input[f"{node.node_id}.full_pose"][:, 3:] / math.pi
            if early:
                pc = pc * 0.0
        o = node_forward_train(node, x, srv["tfs"] if hand else tfs, srv["verts"] if hand else None, fr.repeat_interleave(S),
                               pose_cond=pc, time_code=None if hand else node.frame_latent_encoder(input["idx"]), sync=False, fused=fused)
        f = dict(color=o["color"].reshape(B * P, S, 3), normal=o["normal"].reshape(B * P, S, 3), density=o["density"].reshape(B * P, S), z_vals=z)
        factors.append(f)
        prepare_loss_targets(out, node, B, P, o["x_c"], generator)
        own = composite(net.ctx, [f], [node.class_id])                      # volumetric_render(myfactors) (hold_net.py:86-88)
        for k, v in own.items():
            out[f"{node.node_id}.{k}"] = v
    comp = composite(net.ctx, factors, [nd.class_id for nd in net.nodes.values()])
    out.update(comp)
    R_s = next(iter(net.nodes.values())).bounding_sphere
    out["bg_z_vals"] = (torch.linspace(0.0, 1.0, 32, device=dev) * (1.0 / R_s))[None].expand(B * P, 32)
    out["ray_dirs"], out["cam_loc"], out["index"] = dirs, cam, input["idx"]
    rgb, sem = comp["fg_rgb"], comp["fg_semantics"]
    if getattr(net, "background", None) is not None:                        # hold_net.py:110-134
        bgo = background_forward_train(net.background, comp["bg_weights"], dirs, cam, input["idx"], B, R_s, fused=fused)
        rgb, sem = rgb + bgo["bg_rgb"], sem + bgo["bg_semantics"]
        out["bg_rgb_only"] = bgo["bg_rgb_only"]
    out["rgb"], out["semantics"] = rgb, sem
    if hasattr(net, "step_embedding"):
        net.step_embedding()                                                # hold_net.py:121-122: the BARF counter advances per training forward
    return out


class Loss(torch.nn.Module):
    """hold/loss.py:9-96 with hold/loss_terms.py: L1 rgb, L2 semantics against the one-hot segmentation, opacity sparseness off the
    surface, eikonal (kept only above its lower bound), clamped L1 between the SDF net and the MANO canonical mesh; the reference's
    weights and schedules."""

    def __init__(self, milestone=30000):
        super().__init__()
        self.milestone = milestone

    def forward(self, batch, mo):
        rgb_gt = batch["gt.rgb"].reshape(-1, 3)
        mask_gt = batch["gt.mask"].reshape(-1)
        B = batch["idx"].shape[0]
        scores = torch.ones(B, device=rgb_gt.device)
        valid = torch.ones_like(mask_gt, dtype=torch.float32)
        per_px = lambda n: scores[:, None].repeat(1, n // B).reshape(-1, 1)
        ok = ~torch.any(mo["rgb"].isnan(), dim=1)
        l = (mo["rgb"][ok] - rgb_gt[ok]).abs() * valid[ok][:, None]
        rgb_loss = (l * per_px(l.shape[0])).sum() / (valid[ok].sum() + 1e-6)
        sem = mask_gt.clone().float()                                                # loss_terms.py:70-97
        cls = torch.zeros_like(sem, dtype=torch.long)
        cls[(sem >= 25) & (sem < 100)] = 1
        cls[(sem >= 100) & (sem < 200)] = 2
        cls[sem >= 200] = 3
        onehot = torch.nn.functional.one_hot(cls, len(SEGM_IDS)).float()
        sl = (mo["semantics"] - onehot) ** 2 * valid[:, None]
        sem_loss = (sl * per_px(sl.shape[0])).sum() / valid.sum()
        sparse = 0.0
        for k in [k for k in mo if k.endswith(".index_off_surface")]:
            nid = k.split(".")[0]
            acc, off = mo[f"{nid}.mask_prob"].reshape(-1, 1), mo[k]
            sparse = sparse + (acc[off].abs() * per_px(acc.shape[0])[off]).mean()
        eik = 0.0
        for k in [k for k in mo if k.endswith("grad_theta")]:
            eik = eik + ((mo[k].norm(2, dim=-1) - 1) ** 2).mean()
        mano = 0.0
        for k in [k for k in mo if k.endswith("pts2mano_sdf_cano")]:
            nid = k.split(".")[0]
            p, g = torch.clamp(mo[f"{nid}.pred_sdf"], -0.01, 0.01), torch.clamp(mo[k].detach(), -0.01, 0.01)
            mano = mano + ((p - g).abs() * scores[:, None]).mean()
        progress = min(self.milestone, int(mo.get("step", 0)))
        w_sem = torch.linspace(1.1, 0.1, self.milestone + 1)[progress]
        w_sparse = torch.linspace(0.0, 1.0, self.milestone + 1)[progress]
        d = {"loss/rgb": rgb_loss * 1.0, "loss/sem": sem_loss * w_sem}
        eik = eik * 0.00001
        if float(eik.detach() if torch.is_tensor(eik) else eik) > 0.0008:
            d["loss/eikonal"] = eik
        d["loss/mano_cano"] = mano * 5.0
        d["loss/opacity_sparse"] = sparse * w_sparse
        d["loss"] = sum(d[k] for k in list(d))
        return d


class TrainStep:
    """One data-parallel training step of the foreground model (hold/hold.py:110-137 without the Lightning plumbing): every
    rank takes its share of the step's rays, runs sampler (no grad) -> nodes in training mode -> merge + integrate -> losses,
    back-propagates through the kernels above, then ONE all-reduce over a single flat gradient bucket (shard.allreduce_grads_,
    the only collective of the step: SURVEY §8e) and the optimiser step (Adam, hold.py:79-101).
    The forward is `forward_train` (the reference's training-mode output dict).  Losses of this benchmark step: L1 rgb, L2 semantics
    (loss_terms.py:14-21, :60-70) and the eikonal term (volsdf_utils.py:19-48; loss.py:83-87); the full reference loss incl. the
    kaolin-target terms (mano_cano, opacity_sparse) is `Loss` (pinned to the reference's module, tests/test_cpu_loss.py) on the
    same output dict once the canonical meshes are attached to the nodes.  fused=True: the forward's per-point glue on the fused
    kernels (forward_train(fused=True))."""

    def __init__(self, net, lr=1e-4, n_eik=256, group=None, capturable=False, fused=False):
        self.net, self.group, self.n_eik, self.fused = net, group, n_eik, fused
        self.params = [p for p in net.parameters() if p.requires_grad]
        self.opt = torch.optim.Adam(self.params, lr=lr, capturable=capturable)
        self._graph = None

    # ---- the step as ONE CUDA graph.  The step is ~1 200 small launches on 1 280 rays (packing, sampler rounds, ~70 matrix
    # products, pointwise kernels, Adam): host-bound when launched one by one.  Nothing in it depends on the host (no syncs, no
    # data-dependent control flow: the sampler's convergence gate lives on the device), so after warm-up -- workspaces grown,
    # allocator warm -- it is captured once and replayed; inputs are copied into the captured tensors.
    def capture(self, input, gt_rgb, gt_mask, warmup=3):
        assert self.opt.defaults.get("capturable", False), "TrainStep(..., capturable=True) for graph capture"
        self._static = {k: (v.clone() if torch.is_tensor(v) else v) for k, v in input.items()}
        self._leaf_of = {k: v for k, v in input.items() if torch.is_tensor(v) and v.requires_grad}
        for k, v in self._leaf_of.items():            # pose leaves the caller optimises stay the caller's tensors
            self._static[k] = v
        self._gt = (gt_rgb.clone(), gt_mask.clone())
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(warmup):
                self.step(self._static, *self._gt)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self._graph = torch.cuda.CUDAGraph()
        self.opt.zero_grad(set_to_none=False)
        with torch.cuda.graph(self._graph):
            self._loss, self._parts = self.step(self._static, *self._gt, zero=True)
        return self

    def replay(self, input=None, gt_rgb=None, gt_mask=None):
        """One captured step; new batch contents (same shapes) are copied into the captured tensors first."""
        if input is not None:
            for k, v in input.items():
                if torch.is_tensor(v) and k not in self._leaf_of:
                    self._static[k].copy_(v)
        if gt_rgb is not None:
            self._gt[0].copy_(gt_rgb)
        if gt_mask is not None:
            self._gt[1].copy_(gt_mask)
        self._graph.replay()
        return self._loss, self._parts

    def forward_loss(self, input, gt_rgb, gt_mask, generator=None):
        out = forward_train(self.net, input, generator, fused=self.fused)
        B = input["uv"].shape[0]
        eik = [((out[k].norm(2, dim=-1) - 1) ** 2).mean() for k in out if k.endswith("grad_theta")]
        if not eik:   # no canonical meshes attached to the nodes: the global branch (volsdf_utils.py:36-43), uniform in [-0.3, 0.3]^3
            eik = [((compute_gradient_samples(None, node, self.n_eik, None, B, generator=generator).norm(2, dim=-1) - 1) ** 2).mean()
                   for node in self.net.nodes.values()]
        rgb, sem = out["rgb"], out["semantics"]
        valid = gt_rgb.shape[0]
        loss_rgb = (rgb - gt_rgb).abs().sum() / (valid + 1e-6)
        loss_sem = ((sem - gt_mask) ** 2).mean()
        loss_eik = sum(eik) * 1e-5
        return loss_rgb + loss_sem + loss_eik, dict(rgb=loss_rgb.detach(), sem=loss_sem.detach(), eikonal=loss_eik.detach())

    def step(self, input, gt_rgb, gt_mask, generator=None, zero=True):
        from . import shard

        if zero:
            for p in self.params:                      # in place (captured graphs need stable gradient tensors)
                if p.grad is not None:
                    p.grad.zero_()
        loss, parts = self.forward_loss(input, gt_rgb, gt_mask, generator)
        loss.backward()
        shard.allreduce_grads_(self.params, group=self.group, average=True)
        torch.nn.utils.clip_grad_norm_(self.params, 0.5)      # train.py:30 gradient_clip_val=0.5, after the reduction
        self.opt.step()
        return loss.detach(), parts
