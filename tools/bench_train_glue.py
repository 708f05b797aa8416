"""The training step with the per-point glue as torch ops (fused=False) against the fused glue kernels (fused=True), on the workload of
`bench.py --config train`: 10 frames x 128 pixels, right hand + object + NeRF++ background, per-frame pose leaves.

Each arm runs eager (TrainStep.step) and as one CUDA graph (TrainStep.capture / replay), in one process: first the two eager arms, then
(with the eager models released) the two graphs, each pair alternating in `--reps` rounds of `--steps` steps.  Each step is timed on
its own: host clock, device synchronised before and after, gc.collect() between steps outside the clock (a step's autograd graph is
otherwise freed whenever the cycle collector next runs, and two full-size models then run out of memory).  Before any timing the two
arms take one eager step from the same weights and batch and their losses and gradients are compared.  A separate torch.profiler run counts the CUDA
kernels of one eager step of each arm.  Prints one JSON line and writes it to --out.

    python tools/bench_train_glue.py --out /tmp/bench_train_glue.json"""
import argparse
import gc
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import bench


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True, timeout=10).stdout.strip()
    return {"nvidia_smi": q, "torch_device": torch.cuda.get_device_name(0)}


def make(ctx, dev, fused, capturable):
    """a fresh model (same seeds -> same initial weights), its batch with its own pose leaves, and its TrainStep"""
    from hold_b200 import capi, scene_io, synth, train
    from hold_b200.model import HOLDNet

    Bf, px = 10, 128
    sc = synth.make_scene(H=bench.H, W=bench.W, S=bench.S, nodes=bench.NODES, B=Bf, seed=0)
    for nid in sc.node_ids:
        sc.beta[nid] = torch.tensor(bench.BETA)
    fg = scene_io.build_net(sc, ctx, capi.MLP_TC)
    bg, _, _ = scene_io.build_background(sc, ctx, mlp_mode=capi.MLP_TC)
    net = HOLDNet(ctx, dict(fg.nodes), background=bg)
    gen = torch.Generator().manual_seed(100)
    ids = torch.stack([torch.randperm(bench.H * bench.W, generator=gen)[:px] for _ in range(Bf)])
    inp = scene_io.scene_input(sc, dev)
    inp["uv"] = torch.gather(inp["uv"], 1, ids.to(dev)[:, :, None].expand(-1, -1, 2)).contiguous()
    leaves = []
    for k in list(inp):
        if torch.is_tensor(inp[k]) and inp[k].is_floating_point() and any(k.endswith(s) for s in (".full_pose", ".transl", ".global_orient")):
            inp[k] = inp[k].clone().requires_grad_(True)
            leaves.append(inp[k])
    R = Bf * px
    gt_rgb = torch.rand(R, 3, device=dev, generator=torch.Generator(device=dev).manual_seed(7))
    gt_mask = torch.zeros(R, 4, device=dev)
    gt_mask[:, 0] = 1.0
    ts = train.TrainStep(net, capturable=capturable, fused=fused)
    ts.params = ts.params + leaves
    return dict(net=net, inp=inp, gt=(gt_rgb, gt_mask), ts=ts, R=R)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10, help="steps per timed window")
    ap.add_argument("--reps", type=int, default=5, help="alternating rounds of the four variants")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import __graft_entry__ as g

    g.build()
    from hold_b200 import capi

    assert torch.cuda.is_available(), "bench_train_glue measures on the GPU"
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    ctx = capi.Context(0)
    info = card()

    # ---- agreement of the two arms: one eager step from the same weights, batch and eikonal samples
    arms = {f: make(ctx, dev, f, False) for f in (False, True)}
    chk = {}
    for f, a in arms.items():
        torch.manual_seed(11)
        loss, parts = a["ts"].step(a["inp"], *a["gt"])
        torch.cuda.synchronize()
        ctx.check()
        chk[f] = (loss.item(), [p.grad.detach().clone() for p in a["ts"].params])
        gc.collect()
    loss_d = abs(chk[True][0] - chk[False][0]) / abs(chk[False][0])
    worst, n_cmp = 0.0, 0
    for a_, b_ in zip(chk[True][1], chk[False][1]):
        m = b_.abs().max().item() if b_.numel() else 0.0
        if m > 0:
            worst = max(worst, (a_ - b_).abs().max().item() / m)
            n_cmp += 1
    agree = {"loss_rel_diff": loss_d, "worst_grad_rel_diff": worst, "grad_tensors_compared": n_cmp}
    print("agreement", agree, flush=True)
    assert loss_d < 1e-4 and worst < 1e-3, f"the arms disagree: {agree}"

    # ---- eager: the two arms alternating
    def rounds(var):
        times = {k: [] for k in var}
        for _ in range(args.reps):
            for k, fn in var.items():
                ms = []
                for _ in range(args.steps):
                    gc.collect()     # outside the clock: the step's autograd graphs are freed now, not at an arbitrary later step
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    fn()
                    torch.cuda.synchronize()
                    ms.append(1e3 * (time.perf_counter() - t0))
                times[k].append(statistics.mean(ms))
        ctx.check()
        return times

    for a in arms.values():
        for _ in range(args.warmup):
            a["ts"].step(a["inp"], *a["gt"])
            gc.collect()
    times = rounds({("eager", f): (lambda a=a: a["ts"].step(a["inp"], *a["gt"])) for f, a in arms.items()})
    peak = {"eager_two_models_gib": torch.cuda.max_memory_allocated() / 2**30}
    print("eager ms per step", {f"{'fused' if k[1] else 'torch_glue'}": v for k, v in times.items()}, flush=True)

    # ---- kernels per eager step (profiler run of its own)
    from torch.profiler import ProfilerActivity, profile

    kern = {}
    for f in (False, True):
        a = arms[f]
        l0 = ctx.launches
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            a["ts"].step(a["inp"], *a["gt"])
            torch.cuda.synchronize()
        lib_launches = ctx.launches - l0
        names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
        copies = sum(1 for n in names if "memcpy" in n.lower() or "memset" in n.lower())
        kern["fused" if f else "torch_glue"] = {"cuda_kernels": len(names) - copies, "memcpy_memset": copies, "libhold_b200_launches": lib_launches}
    print("kernels per eager step", kern, flush=True)

    # ---- CUDA graphs: the eager models are released first (each captured step keeps its own memory pool)
    del arms, a
    gc.collect()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    graphs = {}
    for f in (False, True):
        a = make(ctx, dev, f, True)
        a["ts"].capture(a["inp"], *a["gt"], warmup=max(3, args.warmup))
        a["ts"].replay()
        graphs[("graph", f)] = a
    torch.cuda.synchronize()
    ctx.check()
    times.update(rounds({k: (lambda a=a: a["ts"].replay()) for k, a in graphs.items()}))
    peak["graph_two_models_gib"] = torch.cuda.max_memory_allocated() / 2**30

    res = {"what": "TrainStep, torch glue (fused=False) vs fused glue kernels (fused=True); ms per step", "card": info,
           "workload": "bench.py --config train: 10 frames x 128 px, right hand + object + NeRF++ background, pose leaves, eikonal 256/frame",
           "timing": f"host clock around each step, device-synchronised before and after (gc.collect() between steps, not timed); per mode the two arms alternate in {args.reps} rounds of {args.steps} steps (rounds: mean ms per step of each round); {args.warmup} warm-up steps",
           "agreement": agree, "kernels_per_eager_step": kern, "peak_allocated": peak}
    for (mode, f), ts_ in times.items():
        res[f"{mode}_{'fused' if f else 'torch_glue'}_ms"] = {"median": statistics.median(ts_), "min": min(ts_), "max": max(ts_), "rounds": ts_}
    for mode in ("eager", "graph"):
        res[f"{mode}_speedup"] = res[f"{mode}_torch_glue_ms"]["median"] / res[f"{mode}_fused_ms"]["median"]
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
