"""CPU-only, SURVEY §8f rank 4.  The oracle's restatement of the reference's Cython MISE (oracle/mise_oracle.py, the reference's
own octree) is pinned to a run of the reference's compiled module recorded in profiles/r02_bench_aux.jsonl; the MISE
restatement the CUDA kernels run (hold_b200/csrc/mise_phases.h, compiled for the host) is held to the oracle round by round
and bit for bit."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import mise_oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _host():
    out = os.path.join(ROOT, "tests", "_build", "libmise_host.so")
    src = os.path.join(ROOT, "tests", "host", "mise_host.cpp")
    hdr = os.path.join(ROOT, "hold_b200", "csrc", "mise_phases.h")
    if not os.path.exists(out) or os.path.getmtime(out) < max(os.path.getmtime(src), os.path.getmtime(hdr)):
        os.makedirs(os.path.dirname(out), exist_ok=True)
        subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", out, src], check=True)
    lib = C.CDLL(out)
    lib.mise_host_create.restype = C.c_void_p
    lib.mise_host_create.argtypes = [C.c_int, C.c_int, C.c_float]
    lib.mise_host_query.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    lib.mise_host_update.argtypes = [C.c_void_p, C.c_void_p]
    lib.mise_host_to_dense.argtypes = [C.c_void_p, C.c_void_p]
    lib.mise_host_destroy.argtypes = [C.c_void_p]
    return lib


def _field(seed):
    rng = np.random.default_rng(seed)
    c = rng.uniform(0.3, 0.7, size=(3, 3))
    r = rng.uniform(0.12, 0.22, size=3)

    def f(pts, R):   # union of three blobs minus a ripple, exact zeros included through quantisation
        x = pts.astype(np.float32) / np.float32(R)
        d = np.min(np.stack([np.linalg.norm(x - c[i].astype(np.float32), axis=1) - np.float32(r[i]) for i in range(3)]), 0)
        v = (d + np.float32(0.02) * np.sin(np.float32(40.0) * x[:, 0])).astype(np.float32)
        return np.round(v * 64) / 64 if seed % 2 else v     # odd seeds: many values exactly on the threshold
    return f


@pytest.mark.parametrize("res0,depth,seed", [(4, 2, 0), (4, 3, 1), (8, 2, 2), (6, 3, 3), (32, 2, 4)])
def test_host_mise_matches_mise_oracle(res0, depth, seed):
    lib = _host()
    f = _field(seed)
    ref = mise_oracle.MISE(res0, depth, 0.0)
    h = lib.mise_host_create(res0, depth, C.c_float(0.0))
    R = res0 << depth
    G = R + 1
    rounds = 0
    while True:
        pr = ref.query()
        buf = np.zeros((G**3, 3), np.int32)
        n = lib.mise_host_query(h, buf.ctypes.data_as(C.c_void_p), C.c_int(G**3))
        assert n == pr.shape[0], f"round {rounds}: {n} vs {pr.shape[0]} points"
        if n == 0:
            break
        mine = buf[:n]
        key = lambda p: (p[:, 0].astype(np.int64) * G + p[:, 1]) * G + p[:, 2]
        assert np.array_equal(np.sort(key(mine)), np.sort(key(pr))), f"round {rounds}: different point sets"
        ref.update(pr, f(pr, R).astype(np.float64))
        vals = f(mine.astype(np.int64), R).astype(np.float32)
        lib.mise_host_update(h, vals.ctypes.data_as(C.c_void_p))
        rounds += 1
    assert rounds >= 2
    dense_ref = ref.to_dense()
    out = np.empty(G**3, np.float32)
    lib.mise_host_to_dense(h, out.ctypes.data_as(C.c_void_p))
    lib.mise_host_destroy(h)
    assert np.array_equal(out.reshape(G, G, G).astype(np.float64), dense_ref)


def test_mise_oracle_reproduces_recorded_reference_run():
    """tools/bench_aux.py row 8f-4a drove the reference's compiled MISE (32 -> 256, threshold 0) with the oracle's SDF net on the
    canonical object of synth.make_scene(H=8, W=8, S=32, seed=4), through the point mapping of utils/meshing.py:24-32, and
    recorded 845 872 SDF queries (profiles/r02_bench_aux.jsonl).  The oracle replays that run: which voxels subdivide in which
    round decides every count, so an error in the marking or subdivision rules moves it."""
    import torch
    from hold_b200 import synth
    from oracle import hold_oracle as O

    torch.set_num_threads(min(8, os.cpu_count() or 1))
    sc = synth.make_scene(H=8, W=8, S=32, nodes=("right", "object"), seed=4)
    v = sc.obj_pts_cano.numpy().astype(np.float32)
    center, scale = (v.min(0) + v.max(0)) * 0.5, (v.max(0) - v.min(0)).max()
    ex = mise_oracle.MISE(32, 3, 0.0)
    per_round = []
    pts = ex.query()
    with torch.no_grad():
        while pts.shape[0] != 0:
            p = (pts.astype(np.float32) / ex.resolution - 0.5) * 1.1
            p = p * scale + center
            vals = O.sdf_mlp(torch.tensor(p).float(), sc.sdf_state["object"])[:, 0].numpy().astype(np.float64)
            per_round.append(pts.shape[0])
            ex.update(pts, vals)
            pts = ex.query()
    print("queries per round", per_round)
    assert sum(per_round) == 845872
