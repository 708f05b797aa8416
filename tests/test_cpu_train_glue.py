"""CPU-only: the training glue the CUDA kernels run (hold_b200/csrc/train_glue_phases.h, compiled for the host) against float64
torch.autograd over the reference's expressions — the normal of extract_features under detached skinning weights and the Laplace
density (normal, density and the gradients w.r.t. g, sdf, the transforms and beta), and the background's 32-sample AbsDensity
integration (outputs and the gradients w.r.t. rgb, sdf and the foreground's bg_weights)."""
import ctypes as C
import os
import subprocess

import pytest
import torch
import torch.nn.functional as F

from hold_b200 import synth
from oracle import hold_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BAR = 2e-5     # the float64 host tests' bar (tests/test_cpu_warp_bwd.py), relative to max(1, max |reference|)


def _lib():
    out = os.path.join(ROOT, "tests", "_build", "libtrain_glue_host.so")
    src = os.path.join(ROOT, "tests", "host", "train_glue_host.cpp")
    hdr = os.path.join(ROOT, "hold_b200", "csrc", "train_glue_phases.h")
    if not os.path.exists(out) or os.path.getmtime(out) < max(os.path.getmtime(src), os.path.getmtime(hdr)):
        os.makedirs(os.path.dirname(out), exist_ok=True)
        subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", out, src], check=True)
    return C.CDLL(out)


_p = lambda t: None if t is None else C.c_void_p(t.data_ptr())


def err(a, b):
    a, b = a.double(), b.double()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1.0)).item()


def normal_density_ref(hand, xc, g, sdf, tfs, beta, cano=None, W=None):
    """float64: normal = normalize(g . J^-1, eps 1e-6) with J = (sum_j w_j tfs_j)[:3,:3] (w detached, 15 nearest canonical vertices)
    or tfs[:3,:3]; density = LaplaceDensity at beta.  xc, g [B,P,3], sdf [B,P]."""
    B, P, _ = g.shape
    if hand:
        w = torch.stack([O.skin_weights_query(xc[b], cano, W)[0] for b in range(B)]).detach()
        J = torch.einsum("bpn,bnij->bpij", w, tfs)[..., :3, :3]
    else:
        J = tfs[:, None, :3, :3].expand(B, P, 3, 3)
    n = F.normalize(torch.einsum("bpi,bpij->bpj", g, torch.linalg.inv(J)), dim=-1, eps=1e-6)
    rho = (1.0 / beta) * (0.5 + 0.5 * sdf.sign() * torch.expm1(-sdf.abs() / beta))
    return n, rho


def _case(hand, beta, seed):
    g_ = torch.Generator().manual_seed(seed)
    B, P = 2, 300
    if hand:
        sc = synth.make_scene(H=4, W=4, S=32, nodes=("right",), B=B, seed=3)
        art = O.scene_articulation(sc)["right"]
        cano, W, tfs = art["cano_verts"].float().contiguous(), art["skin_W"].float().contiguous(), art["tfs"].float().contiguous()
        xc = cano[torch.randint(0, 778, (B, P), generator=g_)] + 0.03 * torch.randn(B, P, 3, generator=g_)
        xc[:, :20] += 1.5                                   # far points: every confidence clamped
    else:
        cano = W = None
        tfs = torch.eye(4).repeat(B, 1, 1)
        for b in range(B):
            tfs[b, :3, :3] = O.axis_angle_to_matrix(torch.randn(1, 3, generator=g_))[0] * (1.1 + 0.3 * b)
            tfs[b, :3, 3] = torch.randn(3, generator=g_)
        xc = torch.randn(B, P, 3, generator=g_)
    g = torch.randn(B, P, 3, generator=g_)
    g[:, 20:30] *= 1e-8                                     # |m| below eps: the clamped branch of F.normalize
    sdf = torch.randn(B, P, generator=g_) * 3 * beta
    sdf[:, 30:40] = 0.0                                     # sign / abs have zero derivative at 0
    dn, drho = torch.randn(B, P, 3, generator=g_), torch.randn(B, P, generator=g_)
    return dict(B=B, P=P, xc=xc.contiguous(), g=g.contiguous(), sdf=sdf.contiguous(), tfs=tfs.contiguous(), cano=cano, W=W, dn=dn, drho=drho)


@pytest.mark.parametrize("beta", [0.1, 0.03, 0.01])
@pytest.mark.parametrize("kind", ["hand", "object"])
def test_normal_density_on_host(kind, beta):
    lib = _lib()
    hand = kind == "hand"
    c = _case(hand, beta, seed=int(beta * 1000) + hand)
    B, P = c["B"], c["P"]
    # ---- float64 autograd
    g64, s64, t64 = c["g"].double().requires_grad_(), c["sdf"].double().requires_grad_(), c["tfs"].double().requires_grad_()
    b64 = torch.tensor(beta, dtype=torch.float64, requires_grad=True)
    n_ref, rho_ref = normal_density_ref(hand, c["xc"].double(), g64, s64, t64, b64, c["cano"].double() if hand else None,
                                        c["W"].double() if hand else None)
    ref_g, ref_s, ref_t, ref_b = torch.autograd.grad((n_ref * c["dn"].double()).sum() + (rho_ref * c["drho"].double()).sum(),
                                                     (g64, s64, t64, b64))
    # ---- the phases
    ld = 25 if hand else 9
    normal, density, stash = torch.full((B, P, 3), float("nan")), torch.full((B, P), float("nan")), torch.full((B * P * ld,), float("nan"))
    assert lib.nd_fwd_host(C.c_int(hand), C.c_int(B), C.c_int(P), _p(c["xc"]), _p(c["g"]), _p(c["sdf"]), _p(c["tfs"]), _p(c["cano"]), _p(c["W"]),
                           C.c_float(beta), _p(normal), _p(density), _p(stash)) == 0
    assert err(normal, n_ref) < BAR and err(density, rho_ref) < BAR, (err(normal, n_ref), err(density, rho_ref))
    tiny = torch.zeros(B, P, dtype=torch.bool)
    tiny[:, 20:30] = True
    for nt in (32, 128):
        d_g, d_s = torch.full((B, P, 3), float("nan")), torch.full((B, P), float("nan"))
        d_t, d_b = torch.full(c["tfs"].shape, float("nan")), torch.full((1,), float("nan"))
        assert lib.nd_bwd_host(C.c_int(hand), C.c_int(nt), C.c_int(B), C.c_int(P), _p(c["g"]), _p(c["sdf"]), C.c_float(beta), _p(stash),
                               _p(c["dn"]), _p(c["drho"]), _p(d_g), _p(d_s), _p(d_t), _p(d_b)) == 0
        assert (d_s[:, 30:40] == 0).all()
        # the bottom row of each transform is the servers' constant [0, 0, 0, s]: no gradient there (hold_inverse_warp_bwd)
        top = d_t[..., :3, :3]
        checks = (("d_g", d_g[~tiny], ref_g[~tiny]), ("d_g |m| < eps", d_g[tiny], ref_g[tiny]), ("d_sdf", d_s, ref_s),
                  ("d_tfs", top, ref_t[..., :3, :3]), ("d_beta", d_b[0], ref_b))
        for name, a, b in checks:
            e = err(a, b)
            print(f"{kind} beta={beta} nt={nt} {name}: {e:.2e}")
            assert e < BAR, f"{kind} beta={beta} nt={nt} {name}: {e:.2e}"
        assert (d_t[..., 3, :] == 0).all() and (d_t[..., :3, 3] == 0).all()


def test_normal_density_without_seeds_on_host():
    """NULL seeds: d_normal absent -> d_g and d_tfs are 0; d_density absent -> d_sdf and d_beta are 0."""
    lib = _lib()
    c = _case(True, 0.1, seed=7)
    B, P = c["B"], c["P"]
    normal, density, stash = torch.empty(B, P, 3), torch.empty(B, P), torch.empty(B * P * 25)
    lib.nd_fwd_host(C.c_int(1), C.c_int(B), C.c_int(P), _p(c["xc"]), _p(c["g"]), _p(c["sdf"]), _p(c["tfs"]), _p(c["cano"]), _p(c["W"]),
                    C.c_float(0.1), _p(normal), _p(density), _p(stash))
    d_g, d_s, d_t, d_b = torch.empty(B, P, 3), torch.empty(B, P), torch.empty(c["tfs"].shape), torch.empty(1)
    lib.nd_bwd_host(C.c_int(1), C.c_int(64), C.c_int(B), C.c_int(P), _p(c["g"]), _p(c["sdf"]), C.c_float(0.1), _p(stash), None, None,
                    _p(d_g), _p(d_s), _p(d_t), _p(d_b))
    assert (d_g == 0).all() and (d_s == 0).all() and (d_t == 0).all() and (d_b == 0).all()


def bg_integrate_ref(z, sdf, rgb, fgw):
    """float64, the torch path of background_forward_train: z [32] flipped depths, sdf [R,32], rgb [R,32,3], fgw [R]."""
    R = sdf.shape[0]
    dens = sdf.abs()
    dists = torch.cat([(z[:-1] - z[1:])[None].expand(R, -1), torch.full((R, 1), 1e10, dtype=sdf.dtype)], -1)
    fe = dists * dens
    w = (1 - torch.exp(-fe)) * torch.exp(-torch.cumsum(torch.cat([torch.zeros(R, 1, dtype=sdf.dtype), fe[:, :-1]], -1), -1))
    only = (w[:, :, None] * rgb).sum(1)
    sem = torch.zeros(R, 4, dtype=sdf.dtype)
    sem[:, 0] = 1.0
    return fgw[:, None] * only, only, fgw[:, None] * sem


@pytest.mark.parametrize("ld", [1, 5])
def test_background_integration_on_host(ld):
    lib = _lib()
    g_ = torch.Generator().manual_seed(ld)
    R, R_s = 97, 3.0
    z = torch.flip(torch.linspace(0.0, 1.0, 32) * (1.0 / R_s), dims=[-1]).contiguous()
    sdf = (torch.rand(R, 32, generator=g_) * 100.0) * torch.sign(torch.randn(R, 32, generator=g_))   # fe = dist * |sdf| ~ 0 .. 1
    sdf[0] = 0.0                                                                                     # transparent ray
    sdf[1:, 5] = 0.0                                                                                 # zero derivative of abs at 0
    sdf[2, 3:] = 1e4                                                                                 # opaque early
    rgb, fgw = torch.rand(R, 32, 3, generator=g_), torch.rand(R, generator=g_)
    seeds = [torch.randn(R, 3, generator=g_), torch.randn(R, 3, generator=g_), torch.randn(R, 4, generator=g_)]
    s64, c64, w64 = sdf.double().requires_grad_(), rgb.double().requires_grad_(), fgw.double().requires_grad_()
    outs = bg_integrate_ref(z.double(), s64, c64, w64)
    ref = torch.autograd.grad(sum((o * s.double()).sum() for o, s in zip(outs, seeds)), (s64, c64, w64))
    col = torch.zeros(R * 32, ld)
    col[:, 0] = sdf.reshape(-1)
    col = col.contiguous()
    got = [torch.full((R, 3), float("nan")), torch.full((R, 3), float("nan")), torch.full((R, 4), float("nan"))]
    assert lib.bg_fwd_host(C.c_int(R), _p(z), _p(col), C.c_int(ld), _p(rgb), _p(fgw), *[_p(t) for t in got]) == 0
    for name, a, b in zip(("bg_rgb", "bg_rgb_only", "bg_semantics"), got, outs):
        assert err(a, b) < BAR, (name, err(a, b))
    d_rgb, d_sdf, d_w = torch.full((R, 32, 3), float("nan")), torch.full((R, 32), float("nan")), torch.full((R,), float("nan"))
    assert lib.bg_bwd_host(C.c_int(R), _p(z), _p(col), C.c_int(ld), _p(rgb), _p(fgw), *[_p(s) for s in seeds], _p(d_rgb), _p(d_sdf), _p(d_w)) == 0
    assert (d_sdf[1:, 5] == 0).all()
    for name, a, b in (("d_sdf", d_sdf, ref[0]), ("d_rgb", d_rgb, ref[1]), ("d_fg_bg_weights", d_w, ref[2])):
        e = err(a, b)
        print(f"background ld={ld} {name}: {e:.2e}")
        assert e < BAR, f"{name}: {e:.2e}"
    # seeds may be absent: only bg_rgb_only seeded -> no gradient to the foreground's weights
    lib.bg_bwd_host(C.c_int(R), _p(z), _p(col), C.c_int(ld), _p(rgb), _p(fgw), None, _p(seeds[1]), None, _p(d_rgb), _p(d_sdf), _p(d_w))
    assert (d_w == 0).all()


def test_background_integration_nearly_constant_colour_on_host():
    """the regime of the background nets at initialisation: tiny |sdf| (the first 31 samples carry ~1e-4 of the weight each, the
    last one the rest) and nearly constant colour, where d sdf is a small difference of large terms.  Held to float64 relative to
    its own largest entry (torch's float32 autograd of the same expression is at ~4e-4 here)."""
    lib = _lib()
    g_ = torch.Generator().manual_seed(21)
    R, R_s = 64, 3.0
    z = torch.flip(torch.linspace(0.0, 1.0, 32) * (1.0 / R_s), dims=[-1]).contiguous()
    sdf = (0.01 + 0.015 * torch.rand(R, 32, generator=g_)).contiguous()
    rgb = (0.5 + 1e-3 * torch.randn(R, 32, 3, generator=g_)).contiguous()
    fgw = torch.rand(R, generator=g_)
    seeds = [torch.randn(R, 3, generator=g_), torch.randn(R, 3, generator=g_), torch.randn(R, 4, generator=g_)]
    s64, c64, w64 = sdf.double().requires_grad_(), rgb.double().requires_grad_(), fgw.double().requires_grad_()
    outs = bg_integrate_ref(z.double(), s64, c64, w64)
    ref = torch.autograd.grad(sum((o * s.double()).sum() for o, s in zip(outs, seeds)), (s64, c64, w64))
    d_rgb, d_sdf, d_w = torch.empty(R, 32, 3), torch.empty(R, 32), torch.empty(R)
    assert lib.bg_bwd_host(C.c_int(R), _p(z), _p(sdf), C.c_int(1), _p(rgb), _p(fgw), *[_p(s) for s in seeds], _p(d_rgb), _p(d_sdf), _p(d_w)) == 0
    e = ((d_sdf.double() - ref[0]).abs().max() / ref[0].abs().max()).item()
    print(f"background, nearly constant colour: d_sdf {e:.2e} of its largest entry")
    assert e < BAR, e
