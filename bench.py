#!/usr/bin/env python
"""bench.py — rays/s of the HOLD foreground hot path (SURVEY.md §8d metric) on N B200s.

One "step" = one 512x512 frame (262 144 rays) of BASELINE.json configs[1] (right hand + rigid object,
"128 samples/ray" = N_samples_eval 128 / N_samples 64 / N_samples_extra 32, density beta 0.03 so that the
error-bound sampler runs all 5 rounds — the worst case) through hold_render_fg: rays -> 5 sampler rounds
(inverse LBS + SDF net on 128 new samples/ray/round) -> shading of the 98 final samples (SDF + gradient +
feature, skinning Jacobian, colour net, density) -> n-way merge + volume integration, for every node.

  python bench.py --gpus N --steps K --warmup W            # ours (torchrun for N > 1)
  python bench.py ... --dump-outputs DIR                   # + the last timed step's outputs as DIR/<name>.npy
  python bench.py --impl reference [--steps K]             # the reference algorithm on the host CPU cores

Rays shard over ranks with no data-path collective (render.py has no gradients, SURVEY D4): each rank renders
its own frames -> "scaling": "weak".  Timing: CUDA events around exactly K steps, barrier + synchronize on
both sides, max over ranks.  Every step's inputs are 3.3 GB of per-sample work (>> L2), so L2 is cold for the
streamed data by construction; the weights (a few MB) are meant to be L2-resident.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H = W = 512
S = 128
BETA = 0.03
NODES = ("right", "object")
# algorithmic MACs (SURVEY §8d): SDF net 524 544 / point, of which the sampler rounds need the sdf head only
MAC_SDF_FULL = 39 * 256 + 2 * 256 * 256 + 256 * 217 + 4 * 256 * 256 + 256 * 257
MAC_SDF_HEAD = MAC_SDF_FULL - 256 * 256          # no feature rows of lin8
MAC_GRAD = 459_008                               # reverse-mode count of d sdf / d x (SURVEY §8d)
MAC_RGB = {"right": 266_496, "left": 266_496, "object": 274_688}


def flops_per_ray(rounds: int, nodes=NODES, n_eval=S, s_final=S // 2 + S // 4 + 2) -> float:
    """SURVEY §8d: F = r * N_eval * F_sdf + S_f * (F_sdf + F_grad + F_rgb), summed over nodes."""
    tot = 0.0
    for nid in nodes:
        tot += rounds * n_eval * 2 * MAC_SDF_FULL + s_final * 2 * (MAC_SDF_FULL + MAC_GRAD + MAC_RGB[nid])
    return tot


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops", 1590.0), d.get("bf16_tflops_sustained", 1400.0), "measured"
    return 1590.0, 1400.0, "fallback"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.rows = index, threading.Event(), []

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag.is_set():
            try:
                o = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                   capture_output=True, text=True, timeout=5).stdout.strip()
                if o:
                    self.rows.append([x.strip() for x in o.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": int(self.rows[0][1]) if self.rows[0][1].isdigit() else None,
                "reasons": reasons, "samples": len(self.rows)}


def make_scene(seed=0, H_=H, W_=W):
    from hold_b200 import synth

    sc = synth.make_scene(H=H_, W=W_, S=S, nodes=NODES, B=1, seed=seed)
    for nid in sc.node_ids:
        sc.beta[nid] = torch.tensor(BETA)
    return sc


def _cpu_worker(rank, n_workers, threads, n_rays, repeats, barrier, q):
    """One worker of the CPU arm: its own disjoint 512-ray chunks of the frame, `threads` torch threads."""
    import torch as th

    th.set_num_threads(threads)
    sys.path.insert(0, ROOT)
    from oracle import hold_oracle as O

    sc2 = make_scene(0)
    g = th.Generator().manual_seed(11)
    ids_all = th.randperm(H * W, generator=g)[: n_rays * n_workers]
    ids = th.sort(ids_all[rank * n_rays:(rank + 1) * n_rays]).values
    O.render_scene(sc2, ray_ids=ids[:64], chunk=64)  # warm-up (allocator, thread pool)
    barrier.wait()
    t0 = time.perf_counter()
    for _ in range(repeats):
        O.render_scene(sc2, ray_ids=ids, chunk=512)
    q.put((rank, time.perf_counter() - t0))


def usable_cpus() -> int:
    """Hardware threads this process may actually use: scheduler affinity, capped by the cgroup CPU quota (a container on a
    128-thread host may own far fewer; os.cpu_count() does not know)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(float(quota) / float(period))))
    except Exception:
        pass
    return max(1, n)


def cpu_reference_rays_per_s(n_rays_per_worker: int = 1024, repeats: int = 1, threads: int | None = None, workers: int | None = None):
    """The reference's algorithm (oracle port, pinned to the reference modules by oracle/ref_harness.py) on ALL host cores:
    rays are independent, so the frame's 512-ray chunks (datasets/eval_datasets.py:13) are farmed over `workers` processes of
    `threads` torch threads each (one process tops out at ~16 threads on these small GEMMs: sweep on the round-1 box, 2 x Xeon
    8562Y+: 16 threads 105 rays/s, 32: 89, 64: 56, 128: 0.84).  Wall clock from a common start barrier to the last worker's end."""
    import multiprocessing as mp

    ncpu = usable_cpus()
    threads = threads or int(os.environ.get("HOLD_CPU_THREADS", min(16, ncpu)))
    workers = workers or int(os.environ.get("HOLD_CPU_WORKERS", max(1, ncpu // threads)))
    ctx = mp.get_context("spawn")
    barrier, q = ctx.Barrier(workers + 1), ctx.Queue()
    procs = [ctx.Process(target=_cpu_worker, args=(r, workers, threads, n_rays_per_worker, repeats, barrier, q)) for r in range(workers)]
    for p_ in procs:
        p_.start()
    barrier.wait()
    t0 = time.perf_counter()
    done = [q.get() for _ in procs]
    dt = time.perf_counter() - t0
    for p_ in procs:
        p_.join()
    total = n_rays_per_worker * workers * repeats
    return total / dt, threads * workers, dt, dict(workers=workers, threads_per_worker=threads, rays=total, usable_cpus=ncpu,
                                                    os_cpu_count=os.cpu_count(), slowest_worker_s=max(d for _, d in done))


def _cpu_line(rps, cores, dt, info, steps):
    return {"value": rps, "unit": "rays/s", "cores": cores, "kind": "port",
            "sample": f"{info['rays']} rays of the same 512x512 workload ({info['workers']} processes x {info['threads_per_worker']} threads, "
                      f"disjoint 512-ray chunks, {steps} pass(es); {info.get('usable_cpus')} usable hardware threads of {info.get('os_cpu_count')}) in {dt:.1f} s wall; oracle/hold_oracle.py = torch-CPU fp32 restatement pinned "
                      f"to the reference's own modules (oracle/ref_harness.py; /root/reference cannot travel to the GPU box, hence 'port')"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    reps = max(1, args.steps)
    # one 512-ray chunk per worker and step: ~5 s per step on the GPU box's host, so that --steps 20 ends within a few minutes
    rps, cores, dt, info = cpu_reference_rays_per_s(512, repeats=reps)
    line = {
        "impl": "reference", "metric": "rays/sec (128 samples/ray)", "value": rps, "unit": "rays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / reps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "configs[1]: right hand + rigid object, 512x512 frame, 128 samples/ray (N_eval 128, N 64, extra 32), beta 0.03 -> 5 sampler rounds",
                   "sample": f"{info['rays'] // reps} rays of the frame per step, 512-ray chunks over {info['workers']} processes x {info['threads_per_worker']} threads"},
        "cpu_baseline": _cpu_line(rps, cores, dt, info, reps),
        "e2e": {"value": rps, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def ncu_traffic_bytes():
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant launch from the newest committed ncu --set full capture
    (profiles/r*_ncu_k_mlp_tc0*_raw.csv), or None."""
    import csv
    import glob

    cands = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_k_mlp_tc0*raw.csv")))
    for path in reversed(cands):
        try:
            rows = list(csv.reader(open(path)))
            hdr, units = rows[0], rows[1]
            for r in rows[2:]:
                d = dict(zip(hdr, r))
                if "k_mlp_tc" not in d.get("Kernel Name", ""):
                    continue
                tot = 0.0
                for k in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                    u = units[hdr.index(k)].lower()
                    mult = {"byte": 1.0, "kbyte": 1e3, "mbyte": 1e6, "gbyte": 1e9}[u]
                    tot += float(d[k]) * mult
                return tot, os.path.basename(path)
        except Exception:
            continue
    return None, None


def run_train(args):
    """SURVEY C5 / BASELINE configs[4]: one training step = 10 frames x 128 pixels per rank (parser.py:26,87-89) through sampler ->
    nodes in training mode (forward + backward incl. the second-order path) -> merge + integrate -> background -> losses -> ONE flat-bucket
    all-reduce of every gradient -> Adam.  Prints its own JSON line (metric: training rays/s); weak scaling (rays per rank fixed)."""
    import __graft_entry__ as g

    rank, local_rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    if rank == 0:
        g.build()
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_

        dist = dist_
        dist.init_process_group("nccl", device_id=dev)
        dist.barrier()
    from hold_b200 import capi, scene_io, synth, train

    ctx = capi.Context(local_rank)
    Bf, px = 10, 128
    sc = synth.make_scene(H=H, W=W, S=S, nodes=NODES, B=Bf, seed=0)
    for nid in sc.node_ids:
        sc.beta[nid] = torch.tensor(BETA)
    from hold_b200.model import HOLDNet

    fg = scene_io.build_net(sc, ctx, capi.MLP_TC)
    bg, _, _ = scene_io.build_background(sc, ctx, mlp_mode=capi.MLP_TC)
    net = HOLDNet(ctx, dict(fg.nodes), background=bg)      # the whole model: both nodes + the NeRF++ background
    gen = torch.Generator().manual_seed(100 + rank)
    ids = torch.stack([torch.randperm(H * W, generator=gen)[:px] for _ in range(Bf)])          # this rank's pixels of every frame
    inp = scene_io.scene_input(sc, dev)
    inp["uv"] = torch.gather(inp["uv"], 1, ids.to(dev)[:, :, None].expand(-1, -1, 2)).contiguous()
    pose_leaves = []
    for k in list(inp):   # per-frame poses as leaves: the step differentiates through inverse skinning and the pose servers
        if torch.is_tensor(inp[k]) and inp[k].is_floating_point() and any(k.endswith(sfx) for sfx in (".full_pose", ".transl", ".global_orient")):
            inp[k] = inp[k].clone().requires_grad_(True)
            pose_leaves.append(inp[k])
    R = Bf * px
    gt_rgb = torch.rand(R, 3, device=dev, generator=torch.Generator(device=dev).manual_seed(7))
    gt_mask = torch.zeros(R, 4, device=dev)
    gt_mask[:, 0] = 1.0
    ts = train.TrainStep(net, group=None, capturable=args.graph)
    ts.params = ts.params + pose_leaves          # pose gradients ride in the same flat bucket
    n_grad = sum(p.numel() for p in ts.params)

    def sync_all():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    graph_note = "eager launches"
    run = lambda: ts.step(inp, gt_rgb, gt_mask)
    if not args.graph:
        for _ in range(max(1, args.warmup)):
            loss, parts = ts.step(inp, gt_rgb, gt_mask)
        sync_all()
        ctx.check()
        l0 = ctx.launches
        loss, parts = ts.step(inp, gt_rgb, gt_mask)
        launches_per_step = ctx.launches - l0
    else:
        # no eager step on the default stream before the capture: the parameters' AccumulateGrad nodes would be tied to the legacy
        # stream, which a capturing stream may not wait on; capture() warms up on a side stream itself
        try:
            l0 = ctx.launches
            ts.capture(inp, gt_rgb, gt_mask, warmup=max(3, args.warmup))
            launches_per_step = (ctx.launches - l0) // (max(3, args.warmup) + 1)
            run = lambda: ts.replay()
            for _ in range(2):
                run()
            graph_note = "the whole step captured once as ONE CUDA graph and replayed (TrainStep.capture)"
        except Exception as e:   # noqa: BLE001 - a failed capture leaves the CUDA generator / allocator unusable: report and stop
            import traceback

            traceback.print_exc()
            if rank == 0:
                print(json.dumps({"metric": "training rays/sec (forward + backward + gradient all-reduce + Adam)", "unavailable": f"CUDA graph capture failed: {type(e).__name__}: {str(e)[:200]}"}))
            return
    sync_all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        loss, parts = run()
    e1.record()
    sync_all()
    ms = e0.elapsed_time(e1)
    if dist is not None:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    if rank == 0:
        print(json.dumps({
            "metric": "training rays/sec (forward + backward + gradient all-reduce + Adam)", "value": world * R * args.steps / (ms * 1e-3),
            "unit": "rays/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"configs[4] / SURVEY C5: training step, {Bf} frames x {px} pixels per rank, right hand + object, 128 samples/ray, beta {BETA}",
                       "collective": f"one flat-bucket all-reduce of {n_grad} fp32 gradients per step (NCCL)" if world > 1 else "none (1 rank)",
                       "losses": "L1 rgb + L2 semantics + eikonal (256 canonical samples per frame)", "model": "right hand + object + NeRF++ background (32 inverse-sphere samples/ray)",
                       "mlp_mode": "tcgen05 fp16-split x3: hold_linear (activations), hold_wgrad (weight gradients); hold_composite_bwd"},
            "gpu_launches": launches_per_step * args.steps, "launch_mode": graph_note, "loss": float(loss), "loss_terms": {k: float(v) for k, v in parts.items()}}))
    if dist is not None:
        dist.destroy_process_group()


def dump_outputs(out, path):
    """Every tensor of one forward_fg result as <path>/<key>.npy: floating outputs as float32, integer ones as float64 (exact).
    The benchmark's workload gives 48 floats per ray, 50.3 MB for the 512x512 frame."""
    import numpy as np

    arrays = {k: v.detach().cpu() for k, v in out.items() if torch.is_tensor(v)}
    arrays = {k: (v.float() if v.is_floating_point() else v.double()).numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    # H, W and NODES are constants, so the whole result always fits; a larger frame would need a fixed, seeded sample of rays
    assert total <= 64e6, f"outputs of {total / 1e6:.1f} MB exceed the 64 MB a dump may hold"
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, f"{k}.npy"), a)


def positive_int(s):
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError(f"must be at least 1, got {v}")
    return v


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=3, help="timed steps")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default=os.environ.get("HOLD_MLP_MODE", "auto"), choices=["auto", "fp32", "tc"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--graph", action="store_true", help="--config train: capture the step as one CUDA graph and time replays")
    ap.add_argument("--config", default="render", choices=["render", "train"],
                    help="render: BASELINE configs[1] (the driver's line); train: one data-parallel training step (configs[4] / SURVEY C5)")
    ap.add_argument("--no-extras", action="store_true", help="skip the configs[2] (two hands + object) and full-forward (with background) fields")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (rank 0); the inputs are "
                         "seeded, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.config != "render"):
        ap.error("--dump-outputs applies to --impl ours --config render")
    if args.impl == "reference":
        return run_reference(args)
    if args.config == "train":
        return run_train(args)

    import __graft_entry__ as g

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank == 0:
        g.build()
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_

        dist = dist_
        dist.init_process_group("nccl", device_id=dev)
        dist.barrier()
    from hold_b200 import capi, scene_io

    capi.lib()
    ctx = capi.Context(local_rank)
    use_tc = (args.mode == "tc") or (args.mode == "auto" and getattr(capi, "TC_READY", False))
    mode = capi.MLP_TC if use_tc else capi.MLP_FP32
    sc = make_scene(seed=0)           # every rank renders the same scene description; frames differ only by index
    net = scene_io.build_net(sc, ctx, mode)
    inp_host = {k: (v.pin_memory() if torch.is_tensor(v) else v) for k, v in scene_io.scene_input(sc, torch.device("cpu")).items()}
    inp_dev = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in inp_host.items()}
    R = H * W

    def step_resident():
        return net.forward_fg(inp_dev, return_factors=False, want_weights=False)

    out_keys = ("fg_rgb", "mask_prob", "normal", "depth", "fg_semantics", "bg_weights")
    host_out = {k: None for k in out_keys}

    def step_e2e():
        d = {k: (v.to(dev, non_blocking=True) if torch.is_tensor(v) else v) for k, v in inp_host.items()}
        o = net.forward_fg(d, return_factors=False, want_weights=False)
        for k in out_keys:
            host_out[k] = o[k].to("cpu", non_blocking=True)
        return o

    def sync_all():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, steps):
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = ctx.launches
        e0.record()
        for _ in range(steps):
            o = fn()
        e1.record()
        sync_all()
        ms = e0.elapsed_time(e1)
        if dist is not None:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, ctx.launches - l0, o

    for _ in range(max(1, args.warmup)):   # at least one untimed call sizes the workspaces
        o = step_resident()
    torch.cuda.synchronize()
    ctx.check()
    iters = [int(x) for x in o["sampler_iters"].tolist()]
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    ms, launches, o = timed(step_resident, args.steps)
    ms_e2e, _, _ = timed(step_e2e, args.steps)
    if rank == 0:
        clocks.stop_flag.set()
        clocks.join(timeout=2)
    value = world * R * args.steps / (ms * 1e-3)
    e2e_value = world * R * args.steps / (ms_e2e * 1e-3)
    h2d = sum(v.numel() * v.element_size() for v in inp_host.values() if torch.is_tensor(v))
    d2h = sum(v.numel() * v.element_size() for v in host_out.values() if v is not None)

    # ---- roofline of the dominant kernel: the SDF-net launch of one sampler round (R x 128 points), timed live
    P = R * S
    xc = (torch.rand(P, 3, device=dev) - 0.5) * 1.6
    sdf = torch.empty(P, device=dev)
    node = net.nodes["right"]
    import ctypes as C

    def sdf_launch():
        capi.check(capi.lib().hold_sdf_eval(ctx.h, node.slot, P, capi.ptr(xc), None, capi.ptr(sdf), None, None, capi.stream_ptr()))

    for _ in range(2):
        sdf_launch()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n_l = 5
    e0.record()
    for _ in range(n_l):
        sdf_launch()
    e1.record()
    torch.cuda.synchronize()
    k_ms = e0.elapsed_time(e1) / n_l
    burst, sustained, how = measured_peaks()
    k_flops = 2.0 * MAC_SDF_HEAD * P
    achieved = k_flops / (k_ms * 1e-3) / 1e12
    passes = 3 if use_tc else 1
    # dram__bytes_read.sum + dram__bytes_write.sum of this launch, read from the committed ncu --set full capture
    traffic_bytes, traffic_src = ncu_traffic_bytes() if use_tc else (None, None)
    roofline = {
        "bound": "tensor", "achieved": achieved, "peak": burst, "unit": "TFLOP/s", "frac": achieved / burst, "traffic": traffic_bytes, "traffic_source": traffic_src,
        "algorithmic_bytes": 16.0 * P,
        "kernel": "SDF-net launch of one sampler round (262144 x 128 points, sdf head only: 0.918 MFLOP/point algorithmic)",
        "ms_per_launch": k_ms, "peak_source": f"MEASURED_PEAKS.json bf16_tflops ({how}, burst: kernel timed alone)",
        "mma_mode": "tcgen05 kind::f16, fp16 hi/lo split x3 passes (fp32-level operands, fp32 accumulate)" if use_tc else "fp32 FFMA on CUDA cores (no tensor pipe)",
        "frac_of_mode_peak": achieved / (burst / passes) if use_tc else None,
        "whole_step_tflops": world * flops_per_ray(max(iters)) * R * args.steps / (ms * 1e-3) / 1e12,
        "whole_step_frac_of_sustained": world * flops_per_ray(max(iters)) * R * args.steps / (ms * 1e-3) / 1e12 / (sustained * world),
    }

    # ---- extra fields (same JSON line): the full HOLDNet.forward with the NeRF++ background leg on this workload, and
    # BASELINE configs[2] (two hands + object, 289 merged samples).  1 warm-up + 2 timed frames each, this rank only.
    extras = None
    if not args.no_extras and use_tc:
        from hold_b200.model import HOLDNet

        extras = {}
        bg, _, _ = scene_io.build_background(sc, ctx, mlp_mode=mode)
        full = HOLDNet(ctx, dict(net.nodes), background=bg)
        full(inp_dev)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(2):
            full(inp_dev)
        e1.record()
        torch.cuda.synchronize()
        extras["full_forward_with_background_rays_per_s"] = world * R * 2 / (e0.elapsed_time(e1) * 1e-3)
        from hold_b200 import synth

        sc3 = synth.make_scene(H=H, W=W, S=S, nodes=("right", "left", "object"), B=1, seed=0)
        for nid in sc3.node_ids:
            sc3.beta[nid] = torch.tensor(BETA)
        net3 = scene_io.build_net(sc3, ctx, mode)
        inp3 = scene_io.scene_input(sc3, dev)
        o3 = net3.forward_fg(inp3, return_factors=False, want_weights=False)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(2):
            o3 = net3.forward_fg(inp3, return_factors=False, want_weights=False)
        e1.record()
        torch.cuda.synchronize()
        ctx.check()
        extras["configs[2]_two_hands_object_rays_per_s"] = world * R * 2 / (e0.elapsed_time(e1) * 1e-3)
        extras["configs[2]_sampler_rounds"] = [int(x) for x in o3["sampler_iters"].tolist()]
        extras["note"] = "per-rank measurements x world; same 512x512 frame, beta 0.03; background nets on tcgen05"
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    cpu = None
    if not args.no_cpu_baseline and world == 1:
        rps, cores, dt, info = cpu_reference_rays_per_s(512, repeats=1)
        cpu = _cpu_line(rps, cores, dt, info, 1)
    line = {
        "metric": "rays/sec (128 samples/ray)", "value": value, "unit": "rays/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "configs[1]: right hand + rigid object, 512x512 frame per step per GPU, 128 samples/ray (N_eval 128, N 64, extra 32), beta 0.03",
                   "nodes": list(NODES), "rays_per_step_per_gpu": R, "sampler_rounds": iters, "parallelism": f"rays/frames sharded x{world}, no collective",
                   "l2": "per-step working set 3.3 GB of samples >> 126 MB L2 (inputs larger than L2)",
                   "mlp_mode": "tcgen05 fp16-split x3" if use_tc else "fp32 CUDA cores"},
        "e2e": {"value": e2e_value, "unit": "rays/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": launches,
        "clocks": clocks.summary(),
        "roofline": roofline,
        "cpu_baseline": cpu,
        "extras": extras,
        "env": {k: v for k, v in os.environ.items() if k.startswith("HOLD_")},   # the library reads no environment; these steer bench.py only
    }
    print(json.dumps(line))
    if args.dump_outputs:
        dump_outputs(o, args.dump_outputs)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
