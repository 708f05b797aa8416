"""SURVEY §8f rank 4: the GPU MISE + fused-MLP SDF queries against the oracle's restatement of the reference's MISE
(oracle/mise_oracle.py, the reference's own octree) fed with the SAME SDF values round by round -> identical dense grids.  The
oracle's pin to a recorded run of the reference's compiled MISE, and the kernels' restatement against the oracle on the host,
are in tests/test_cpu_mise.py."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def impl_generate_grid_matches_mise_oracle(ctx):
    from hold_b200 import capi, meshing, scene_io, synth
    from oracle import mise_oracle

    dev = torch.device("cuda", 0)
    sc = synth.make_scene(H=8, W=8, S=32, nodes=("right", "object"), seed=4)
    net = scene_io.build_net(sc, ctx, capi.MLP_FP32)
    node = net.nodes["object"]
    func = meshing.node_sdf_func(ctx, node)
    verts = sc.obj_pts_cano.numpy()
    grid, res, gt_scale, gt_center = meshing.generate_grid(ctx, func, verts, 0.0, res_init=8, res_up=2)
    ctx.check()
    # the reference's loop (utils/meshing.py:19-47) with the same SDF function
    ex = mise_oracle.MISE(8, 2, 0.0)
    pts = ex.query()
    rounds = 0
    while pts.shape[0] != 0:
        p = pts.astype(np.float32)
        p = (p / ex.resolution - 0.5) * 1.1
        p = p * gt_scale + gt_center
        vals = func(torch.tensor(p).float().to(dev).contiguous()).cpu().numpy().astype(np.float64)
        ex.update(pts, vals)
        pts = ex.query()
        rounds += 1
    ref = ex.to_dense()
    assert rounds >= 2 and grid.shape == ref.shape == (33, 33, 33)
    assert np.array_equal(grid, ref)
    assert (grid < 0).any() and (grid > 0).any()


def test_generate_grid_matches_mise_oracle(isolated):
    isolated("tests/test_gpu_mise.py", "impl_generate_grid_matches_mise_oracle")
