"""The fused training glue on the GPU (hold_b200/csrc/train_glue.cuh): NormalDensityFn, bg_inputs and BgIntegrateFn against float64
autograd over the oracle, bitwise run-to-run reproducibility, node_forward_train / forward_train with fused=True against the torch
glue (fused=False) on the same inputs, and TrainStep(fused=True) replayed as one CUDA graph.  The host arithmetic of the kernels is
held to float64 autograd in tests/test_cpu_train_glue.py."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
TOL = 1e-4


def rel(a, r):
    a, r = a.detach().double().cpu(), r.detach().double().cpu()
    return ((a - r).abs().max() / r.abs().max().clamp_min(1e-30)).item()


def _node_inputs(ctx, nid):
    """the scene, points and seeds of test_gpu_train.py::test_node_training_forward_backward, with x_c, g = d sdf / d x_c and sdf from
    the float64 oracle"""
    from hold_b200 import capi, scene_io, synth
    from oracle import hold_oracle as O

    sc = synth.make_scene(H=8, W=8, S=32, nodes=("right", "object"), B=2, seed=6, perturb=0.02)
    net = scene_io.build_net(sc, ctx, capi.MLP_TC)
    a = O.scene_articulation(sc)[nid]
    hand = nid != "object"
    g = torch.Generator().manual_seed(5)
    B, P = sc.B, 600
    x = (torch.rand(B, P, 3, generator=g) - 0.5) * 1.2
    fr = torch.arange(B).repeat_interleave(P)
    sds, sdr = ({k: v.double() for k, v in sd.items()} for sd in (sc.sdf_state[nid], sc.rgb_state[nid]))
    r = O.node_forward_train(a["kind"], x.reshape(-1, 3).double(), fr, sds, sdr, sc.beta[nid].double(), a["tfs"].double(),
                             posed_verts=a.get("verts").double() if hand else None, cano_verts=a.get("cano_verts").double() if hand else None,
                             skin_W=a.get("skin_W").double() if hand else None,
                             pose_cond=a["pose_cond"].double() if hand else None, time_code=None if hand else sc.time_code.double())
    dn, drho = torch.randn(B * P, 3, generator=g) * 0.1, torch.randn(B * P, generator=g) * 0.01
    return dict(sc=sc, net=net, node=net.nodes[nid], a=a, hand=hand, B=B, P=P, x=x, fr=fr, xc=r["x_c"].detach().float(), g=r["grad"].detach().float(),
                sdf=r["sdf"].detach().float(), beta=float(sc.beta[nid].abs() + 1e-4), dn=dn, drho=drho)


def normal_density_ref(c):
    """float64 autograd of the reference's expressions on the same (float32-rounded) inputs -> outputs and d (g, sdf, tfs, beta)"""
    B, P, a = c["B"], c["P"], c["a"]
    g64, s64 = c["g"].double().requires_grad_(), c["sdf"].double().requires_grad_()
    t64 = a["tfs"].double().clone().requires_grad_()
    b64 = torch.tensor(c["beta"], dtype=torch.float64, requires_grad=True)
    if c["hand"]:
        from oracle import hold_oracle as O

        xc = c["xc"].double().reshape(B, P, 3)
        w = torch.stack([O.skin_weights_query(xc[b], a["cano_verts"].double(), a["skin_W"].double())[0] for b in range(B)]).detach()
        J = torch.einsum("bpn,bnij->bpij", w, t64)[..., :3, :3].reshape(B * P, 3, 3)
    else:
        J = t64[:, None, :3, :3].expand(B, P, 3, 3).reshape(B * P, 3, 3)
    n = F.normalize(torch.einsum("bi,bij->bj", g64, torch.linalg.inv(J)), dim=1, eps=1e-6)
    rho = (1.0 / b64) * (0.5 + 0.5 * s64.sign() * torch.expm1(-s64.abs() / b64))
    grads = torch.autograd.grad((n * c["dn"].double()).sum() + (rho * c["drho"].double()).sum(), (g64, s64, t64, b64))
    return n.detach(), rho.detach(), grads


def _run_normal_density(c, dev):
    from hold_b200 import train

    g = c["g"].to(dev).requires_grad_()
    s = c["sdf"].to(dev).requires_grad_()
    t = c["a"]["tfs"].float().to(dev).requires_grad_()
    b = torch.tensor(c["beta"], device=dev).requires_grad_()
    n, rho = train.NormalDensityFn.apply(c["node"], c["B"], c["xc"].to(dev), g, s, t, b)
    ((n * c["dn"].to(dev)).sum() + (rho * c["drho"].to(dev)).sum()).backward()
    return n.detach(), rho.detach(), (g.grad, s.grad, t.grad, b.grad)


def _bg_inputs_case(ctx):
    """the scene and rays of test_gpu_train.py::test_background_training; sdf and rgb of the background nets from the float64 oracle"""
    from hold_b200 import capi, scene_io, synth
    from oracle import hold_oracle as O

    sc = synth.make_scene(H=12, W=12, S=32, nodes=("right", "object"), B=2, seed=8)
    sc.intrinsics[:, 0, 2] += 0.37
    sc.intrinsics[:, 1, 2] -= 0.21
    scene_io.build_net(sc, ctx, capi.MLP_TC)
    bg, sdf_sd, rgb_sd = scene_io.build_background(sc, ctx, mlp_mode=capi.MLP_TC)
    dirs, cam = O.camera_rays(sc.uv, sc.extrinsics, sc.intrinsics)
    P = dirs.shape[1]
    dirs, cam = dirs.reshape(-1, 3), cam.unsqueeze(1).repeat(1, P, 1).reshape(-1, 3)
    R = dirs.shape[0]
    g = torch.Generator().manual_seed(3)
    bgw = torch.rand(R, generator=g)
    frame = torch.arange(sc.B).repeat_interleave(P)
    idx = torch.as_tensor(sc.frame_idx)
    R_s = sc.bounding_sphere
    zf = torch.flip(O.uniform_z(0.0, torch.ones(R, 1), 32) * (1.0 / R_s), dims=[-1]).double()
    p4 = O.depth2pts_outside(cam.double()[:, None].repeat(1, 32, 1), dirs.double()[:, None].repeat(1, 32, 1), zf, R_s).reshape(-1, 4)
    fc = bg.frame_latent_encoder.weight.detach().cpu().double()[idx][frame].repeat_interleave(32, 0)
    sd64 = {k: v.double() for k, v in sdf_sd.items()}
    o = O.bg_sdf_mlp(p4, fc, sd64)
    rgb = O.bg_rgb_mlp(dirs.double().repeat_interleave(32, 0), fc, o[:, 1:], {k: v.double() for k, v in rgb_sd.items()})
    seeds = [torch.randn(R, 3, generator=g), torch.randn(R, 3, generator=g), torch.randn(R, 4, generator=g)]
    return dict(bg=bg, R=R, R_s=R_s, dirs=dirs, cam=cam, bgw=bgw, zf=zf[0], p4=p4, sdf=o[:, 0].float(), rgb=rgb.float(), seeds=seeds)


def _run_bg_integrate(c, ctx, dev, ld=257):
    from hold_b200 import train

    col = torch.zeros(c["R"] * 32, ld, device=dev)
    col[:, 0] = c["sdf"].to(dev)
    col.requires_grad_()
    sdf = col[:, 0]                                       # a strided column, as BgSdfFn's output in background_forward_train
    rgb, w = c["rgb"].to(dev).requires_grad_(), c["bgw"].to(dev).requires_grad_()
    outs = train.BgIntegrateFn.apply(ctx, c["R_s"], sdf, rgb, w)
    sum((o * s.to(dev)).sum() for o, s in zip(outs, c["seeds"])).backward()
    return [o.detach() for o in outs], (col.grad[:, 0], rgb.grad, w.grad)


def impl_functions_against_float64(ctx):
    from hold_b200 import train

    dev = torch.device("cuda", 0)
    for nid in ("right", "object"):
        c = _node_inputs(ctx, nid)
        n_ref, rho_ref, ref = normal_density_ref(c)
        n, rho, got = _run_normal_density(c, dev)
        ctx.check()
        en, er = rel(n, n_ref), rel(rho, rho_ref)
        print(f"{nid}: normal {en:.2e} density {er:.2e}")
        assert en < 2e-4 and er < TOL, (nid, en, er)
        for name, a, r in zip(("d_g", "d_sdf", "d_tfs", "d_beta"), got, ref):
            if name == "d_tfs":   # the servers' constant bottom row carries no gradient (hold_inverse_warp_bwd)
                a, r = a[..., :3, :3], r[..., :3, :3]
            e = rel(a, r)
            print(f"{nid}: {name} {e:.2e}")
            assert e < 3e-4, f"{nid} {name}: {e:.2e}"
        assert (got[2][..., 3, :] == 0).all() and (got[2][..., :3, 3] == 0).all()
    c = _bg_inputs_case(ctx)
    emb_pts, emb_view = train.bg_inputs(ctx, c["dirs"].to(dev), c["cam"].to(dev), c["R_s"])
    ctx.check()
    from oracle import hold_oracle as O

    for name, a, r in (("bg_inputs points", emb_pts, O.embed_n(c["p4"], 10)),
                       ("bg_inputs view", emb_view, O.embed_n(c["dirs"].double().repeat_interleave(32, 0), 4))):
        e = (a.cpu().double() - r).abs().max().item()
        print(f"{name}: max |d| {e:.2e}")
        assert e <= TOL, f"{name}: {e:.2e}"
    s64, c64, w64 = c["sdf"].double().requires_grad_(), c["rgb"].double().requires_grad_(), c["bgw"].double().requires_grad_()
    R = c["R"]
    dens = s64.abs().reshape(R, 32)
    dists = torch.cat([(c["zf"][:-1] - c["zf"][1:])[None].expand(R, -1), torch.full((R, 1), 1e10, dtype=torch.float64)], -1)
    fe = dists * dens
    wts = (1 - torch.exp(-fe)) * torch.exp(-torch.cumsum(torch.cat([torch.zeros(R, 1, dtype=torch.float64), fe[:, :-1]], -1), -1))
    only = (wts[:, :, None] * c64.reshape(R, 32, 3)).sum(1)
    sem = torch.zeros(R, 4, dtype=torch.float64)
    sem[:, 0] = 1.0
    outs_ref = (w64[:, None] * only, only, w64[:, None] * sem)
    ref = torch.autograd.grad(sum((o * s.double()).sum() for o, s in zip(outs_ref, c["seeds"])), (s64, c64, w64))
    outs, got = _run_bg_integrate(c, ctx, dev)
    ctx.check()
    for name, a, r in zip(("bg_rgb", "bg_rgb_only", "bg_semantics"), outs, outs_ref):
        e = (a.cpu().double() - r).abs().max().item()
        print(f"background: {name} max |d| {e:.2e}")
        assert e <= TOL, f"{name}: {e:.2e}"
    for name, a, r in zip(("d_sdf", "d_rgb", "d_fg_bg_weights"), got, ref):
        e = rel(a, r)
        print(f"background: {name} {e:.2e}")
        assert e < 3e-4, f"background {name}: {e:.2e}"


def test_functions_against_float64(isolated):
    isolated("tests/test_gpu_train_glue.py", "impl_functions_against_float64")


def test_functions_bitwise_reproducible(ctx):
    """two calls of each Function on the same inputs: outputs and gradients bit for bit (fixed-order sums, no float atomics)"""
    dev = torch.device("cuda", 0)
    for nid in ("right", "object"):
        c = _node_inputs(ctx, nid)
        r1, r2 = _run_normal_density(c, dev), _run_normal_density(c, dev)
        ctx.check()
        assert torch.equal(r1[0], r2[0]) and torch.equal(r1[1], r2[1]), nid
        assert all(torch.equal(a, b) for a, b in zip(r1[2], r2[2])), nid
    c = _bg_inputs_case(ctx)
    r1, r2 = _run_bg_integrate(c, ctx, dev), _run_bg_integrate(c, ctx, dev)
    ctx.check()
    assert all(torch.equal(a, b) for a, b in zip(r1[0], r2[0])) and all(torch.equal(a, b) for a, b in zip(r1[1], r2[1]))


# fused=True against fused=False: bounds at <= 3x the differences measured on a B200 (printed by the tests)
NODE_BOUND = {"out": 7e-7, "grad": 8e-5}      # measured: right 2.4e-7 / 2.8e-5, object 1.2e-7 / 2.8e-5
SCENE_BOUND = {"out": 5e-7, "grad": 7e-5}     # measured: 1.7e-7 / 2.3e-5


@pytest.mark.parametrize("nid", ["right", "object"])
def test_node_forward_train_fused_matches_torch_glue(ctx, nid):
    from hold_b200 import train

    c = _node_inputs(ctx, nid)
    node, a, hand, dev = c["node"], c["a"], c["hand"], torch.device("cuda", 0)
    B, P = c["B"], c["P"]
    g = torch.Generator().manual_seed(9)
    cw, dw, nw = torch.randn(B * P, 3, generator=g), torch.randn(B * P, generator=g) * 0.01, torch.randn(B * P, 3, generator=g) * 0.1
    res = {}
    for fused in (False, True):
        node.zero_grad(set_to_none=True)
        tg = a["tfs"].to(dev).requires_grad_(True)
        pg = a["pose_cond"].to(dev).requires_grad_(True) if hand else None
        cg = c["sc"].time_code.to(dev).clone().requires_grad_(True) if not hand else None
        o = train.node_forward_train(node, c["x"].to(dev), tg, a["verts"].to(dev) if hand else None, c["fr"].to(dev), pose_cond=pg, time_code=cg,
                                     fused=fused)
        ((o["color"] * cw.to(dev)).sum() + (o["density"] * dw.to(dev)).sum() + (o["normal"] * nw.to(dev)).sum()).backward()
        ctx.check()
        grads = {n: p.grad.clone() for n, p in node.named_parameters() if p.grad is not None}
        grads["tfs"] = tg.grad[..., :3, :].clone()
        grads["pose_cond" if hand else "time_code"] = (pg if hand else cg).grad.clone()
        res[fused] = ({k: o[k].detach().clone() for k in ("sdf", "x_c", "feat", "grad", "normal", "color", "density")}, grads)
    (o0, g0), (o1, g1) = res[False], res[True]
    worst_o = max(rel(o1[k], o0[k]) for k in o0)
    for k in o0:
        print(f"{nid}: fused vs torch glue, forward {k}: {rel(o1[k], o0[k]):.2e}")
    assert set(g0) == set(g1), sorted(set(g0) ^ set(g1))
    worst_g = 0.0
    for k in g0:
        if g0[k].abs().max() == 0:
            assert g1[k].abs().max() == 0, k
            continue
        e = rel(g1[k], g0[k])
        worst_g = max(worst_g, e)
        print(f"{nid}: fused vs torch glue, grad {k}: {e:.2e}")
    print(f"{nid}: fused vs torch glue, worst forward {worst_o:.2e}, worst gradient {worst_g:.2e}")
    assert worst_o <= NODE_BOUND["out"] and worst_g <= NODE_BOUND["grad"], (worst_o, worst_g)


def _scene(ctx, seed=5):
    from hold_b200 import capi, scene_io, synth
    from hold_b200.model import HOLDNet

    sc = synth.make_scene(H=8, W=8, S=32, nodes=("right", "object"), B=2, seed=seed)
    sc.intrinsics[:, 0, 2] += 0.37
    net = scene_io.build_net(sc, ctx, capi.MLP_TC)
    bg, _, _ = scene_io.build_background(sc, ctx, mlp_mode=capi.MLP_TC)
    return sc, HOLDNet(ctx, dict(net.nodes), background=bg)


def test_forward_train_fused_matches_torch_glue(ctx):
    """the whole model (two nodes + background): every output of forward_train and every parameter's gradient of a random linear
    functional of the outputs, fused=True against fused=False on the same weights and batch"""
    from hold_b200 import scene_io, train

    dev = torch.device("cuda", 0)
    sc, full = _scene(ctx)
    inp = scene_io.scene_input(sc, dev)
    res = {}
    for fused in (False, True):
        full.zero_grad(set_to_none=True)
        out = train.forward_train(full, inp, fused=fused)
        keys = sorted(k for k, v in out.items() if torch.is_tensor(v) and v.is_floating_point() and v.requires_grad)
        g = torch.Generator(device=dev).manual_seed(2)
        sum((out[k] * torch.randn(out[k].shape, device=dev, generator=g)).sum() for k in keys).backward()
        ctx.check()
        res[fused] = ({k: out[k].detach().clone() for k in keys}, {n: p.grad.clone() for n, p in full.named_parameters() if p.grad is not None})
    (o0, g0), (o1, g1) = res[False], res[True]
    assert set(o0) == set(o1) and set(g0) == set(g1)
    assert {"rgb", "semantics", "bg_rgb_only", "right.normal", "object.fg_rgb"} <= set(o0)
    worst_o = max(rel(o1[k], o0[k]) for k in o0)
    worst_g, worst_name = 0.0, None
    for k in g0:
        if g0[k].abs().max() == 0:
            assert g1[k].abs().max() == 0, k
            continue
        e = rel(g1[k], g0[k])
        if e > worst_g:
            worst_g, worst_name = e, k
    for k in o0:
        print(f"forward_train fused vs torch glue, {k}: {rel(o1[k], o0[k]):.2e}")
    print(f"forward_train fused vs torch glue: worst output {worst_o:.2e}, worst gradient {worst_g:.2e} ({worst_name}), {len(g0)} parameters")
    assert worst_o <= SCENE_BOUND["out"] and worst_g <= SCENE_BOUND["grad"], (worst_o, worst_g, worst_name)


def test_train_step_fused_cuda_graph_replay(ctx):
    """TrainStep(fused=True): the whole step as one CUDA graph gives the losses of step-by-step launches (as
    test_gpu_train.py::test_train_step_cuda_graph_replay for the torch glue)."""
    from hold_b200 import scene_io, train

    dev = torch.device("cuda", 0)
    sc, eager = _scene(ctx)
    inp = scene_io.scene_input(sc, dev)
    R = sc.B * sc.uv.shape[1]
    g = torch.Generator(device=dev).manual_seed(0)
    gt_rgb, gt_mask = torch.rand(R, 3, device=dev, generator=g), torch.zeros(R, 4, device=dev)
    gt_mask[:, 0] = 1.0
    torch.manual_seed(3)
    te = train.TrainStep(eager, lr=1e-4, n_eik=64, fused=True)
    le = [te.step(inp, gt_rgb, gt_mask)[0].item() for _ in range(5)]
    ctx.check()
    _, graphed = _scene(ctx)
    torch.manual_seed(3)
    tg = train.TrainStep(graphed, lr=1e-4, n_eik=64, capturable=True, fused=True)
    tg.capture(inp, gt_rgb, gt_mask, warmup=3)
    lg = [tg.replay()[0].item() for _ in range(2)]
    ctx.check()
    print("fused: eager losses", le, "graph replays (steps 4, 5)", lg)
    # same bound and reasoning as the torch-glue test: the eikonal samples of eager steps 4, 5 and of the replays differ
    assert abs(lg[0] - le[3]) <= 2e-2 * abs(le[3]) and abs(lg[1] - le[4]) <= 2e-2 * abs(le[4]), (le, lg)
    assert lg[1] < lg[0] < le[0], (le, lg)
