"""bench.py --config 3 | 4 | 5: the BASELINE configurations next to the headline one (SURVEY.md §8d), each as one JSON
line with the same contract keys (metric / value / e2e / roofline / cpu_baseline ...).

  3  RAFT flow + LAFC completion, synthetic 480x864 clip, T=20: 19 forward + 19 backward RAFT pairs (20 iterations,
     batches of 4 pairs, CUDA-graph replay) and 38 LAFC calls at 240x432; frames/s = 20 / t. N>1: every rank its own
     clip (pairs and calls are independent per frame pair: no data-path collective), weak scaling.
  4  FGT on a 432x240 T=80 clip: the driver's 16 windows (tool/video_inpainting.py:710-717: t = 13..18 input frames each)
     sharded over the ranks by frames per window (longest-processing-time first); frames/s = 80 / max-over-ranks time
     of a rank's windows; strong scaling (the clip is fixed).
  5  FGT on a 1280x720 T=40 clip: the driver's 8 windows (t = 12..14, 21k-key temporal zones, runtime geometry), sharded
     the same way.

--impl reference runs the CPU oracle port on a bounded sample of the same workload (one RAFT pair + one LAFC call for
config 3, one window for configs 4 / 5) and scales it to the metric's unit.
"""
import argparse
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from fgt_b200 import synth  # noqa: E402

SPECS = {
    3: dict(metric="flow_frames_per_sec_480x864_T20", T=20, H=480, W=864,
            workload="RAFT flow (19+19 pairs, 20 iterations) + LAFC completion (38 calls at 240x432), synthetic 480x864 "
                     "clip T=20, real-shape seeded weights"),
    4: dict(metric="inpainted_frames_per_sec_432x240_T80", T=80, H=240, W=432,
            workload="FGT end-to-end over a synthetic 432x240 T=80 clip: the driver's 16 windows, sharded over the ranks"),
    5: dict(metric="inpainted_frames_per_sec_1280x720_T40", T=40, H=720, W=1280,
            workload="FGT over a synthetic 1280x720 T=40 clip: the driver's 8 windows (window-partition + global-token "
                     "path, runtime geometry), sharded over the ranks"),
}


def _events(fn, steps, warmup, flush, barrier):
    with torch.no_grad():
        for _ in range(warmup):
            fn()
        barrier()
        evs = []
        for _ in range(steps):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            evs.append((a, b))
        barrier()
    return sum(a.elapsed_time(b) for a, b in evs) / steps


def _dominant(recs, reps, peaks):
    agg = {}
    for kern, tag, fl, by, ms, _sc in recs:
        a = agg.setdefault(kern, dict(ms=0.0, flops=0.0, bytes=0.0, n=0))
        a["ms"] += ms / reps
        a["flops"] += fl / reps
        a["bytes"] += by / reps
        a["n"] += 1 / reps
    tot = sum(a["ms"] for a in agg.values())
    kernels = {}
    for k, a in sorted(agg.items(), key=lambda kv: -kv[1]["ms"]):
        e = {"ms_per_step": round(a["ms"], 4), "share": round(a["ms"] / tot, 4), "launches_per_step": round(a["n"])}
        if a["flops"] > 0:
            tf = a["flops"] / (a["ms"] * 1e-3) / 1e12
            e.update(bound="tensor", achieved_tflops=round(tf, 2), frac=round(tf / peaks["tf_sustained"], 4))
        else:
            gbs = a["bytes"] / (a["ms"] * 1e-3) / 1e9
            e.update(bound="hbm", achieved_gbs=round(gbs, 1), frac=round(gbs / peaks["hbm_gbs"], 4))
        kernels[k] = e
    dk, da = max(agg.items(), key=lambda kv: kv[1]["ms"])
    if da["flops"] > 0:
        ach = da["flops"] / (da["ms"] * 1e-3) / 1e12
        roof = {"kernel": dk, "bound": "tensor", "achieved": ach, "peak": peaks["tf_sustained"], "unit": "TFLOP/s",
                "frac": ach / peaks["tf_sustained"], "traffic": None, "peak_source": peaks["source"] + ", sustained bf16",
                "note": "algorithmic FLOPs; 3 MMAs per algorithmic one (split-bf16), ceiling 1/3"}
    else:
        ach = da["bytes"] / (da["ms"] * 1e-3) / 1e9
        roof = {"kernel": dk, "bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": ach / peaks["hbm_gbs"], "traffic": None, "peak_source": peaks["source"]}
    return roof, kernels


def _reference(args, spec, out):
    """CPU oracle port on a bounded sample, scaled to frames/s of the whole workload."""
    import bench
    threads = bench.cpu_threads()
    t0 = time.perf_counter()
    if args.config == 3:
        from oracle import lafc_oracle as LO
        from oracle import raft_oracle as RO
        sd = synth.raft_state_dict(seed=4)
        im1, im2 = synth.raft_inputs(seed=5, H=spec["H"], W=spec["W"])
        lsd = synth.make_state_dict(synth.lafc_param_shapes(), seed=5)
        fl, mk = synth.lafc_inputs(seed=6, H=spec["H"] // 2, W=spec["W"] // 2)
        with torch.no_grad():
            t1 = time.perf_counter()
            RO.raft_forward(sd, im1, im2, iters=20)
            t_pair = time.perf_counter() - t1
            t1 = time.perf_counter()
            LO.lafc_forward({k[4:]: v for k, v in lsd.items()}, fl, mk)
            t_call = time.perf_counter() - t1
        sec = 38 * t_pair + 38 * t_call
        sample = f"1 RAFT pair ({t_pair:.2f} s) + 1 LAFC call ({t_call:.2f} s), scaled to 38 + 38"
    else:
        from fgt_b200 import parallel
        from oracle import fgt_oracle as O
        cfg = dict(synth.CFG_A)
        sd = O.strip_net(synth.make_state_dict(synth.fgt_param_shapes(cfg), seed=1, regime="scaled"))
        sched = parallel.window_schedule(spec["T"])
        tot = sum(len(nb) + len(ref) for _, nb, ref in sched)
        ts = 4 if args.config == 5 else 6
        clip = synth.fgt_inputs(seed=3, t=ts, H=spec["H"], W=spec["W"])
        with torch.no_grad():
            t1 = time.perf_counter()
            O.fgt_forward(sd, *clip)
            per_frame = (time.perf_counter() - t1) / ts
        sec = per_frame * tot
        sample = (f"one T={ts} forward at {spec['W']}x{spec['H']} ({per_frame:.2f} s per input frame), scaled to the "
                  f"{tot} input frames of the clip's {len(sched)} windows (under-counts the T^2 attention term)")
    fps = spec["T"] / sec
    print(json.dumps({
        "impl": "reference", "metric": spec["metric"], "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "weak" if args.config == 3 else "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": spec["workload"]},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "host_cores": os.cpu_count(), "kind": "port",
                         "sample": sample},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": time.perf_counter() - t0,
    }), file=out, flush=True)


def run(args, rank, local_rank, world, out):
    spec = SPECS[args.config]
    if args.impl == "reference":
        if rank == 0:
            _reference(args, spec, out)
        return
    import torch.distributed as dist
    import bench
    from fgt_b200 import lib, parallel
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    peaks = bench.load_peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = bench.ClockSampler(local_rank)
    extra = {}
    if args.config == 3:
        from fgt_b200.lafc_model import Model as LAFC
        from fgt_b200.raft_model import RAFT
        T, H, W = spec["T"], spec["H"], spec["W"]
        raft = RAFT(argparse.Namespace(small=False, mixed_precision=False, alternate_corr=False))
        raft.load_state_dict(synth.raft_state_dict(seed=4))
        raft = raft.to(dev).eval()
        raft.enable_cuda_graph(True)
        lafc = LAFC(synth.CFG_LAFC)
        lafc.load_state_dict(synth.make_state_dict(synth.lafc_param_shapes(), seed=5))
        lafc = lafc.to(dev)
        lafc.net.enable_cuda_graph(True)
        npairs = 2 * (T - 1)
        im1, im2 = synth.raft_inputs(seed=5 + rank, H=H, W=W, n=npairs)          # forward and backward pairs of the clip
        h1, h2 = im1.pin_memory(), im2.pin_memory()
        d1, d2 = h1.to(dev), h2.to(dev)
        fl, mk = synth.lafc_inputs(seed=6 + rank, H=H // 2, W=W // 2)
        hfl, hmk = fl.pin_memory(), mk.pin_memory()
        dfl, dmk = hfl.to(dev), hmk.to(dev)
        rb = 4
        flows_host = torch.empty(npairs, 2, H, W).pin_memory()

        def step(host_io):
            for s in range(0, npairs, rb):
                a, b = (h1[s:s + rb].to(dev, non_blocking=True), h2[s:s + rb].to(dev, non_blocking=True)) if host_io else \
                       (d1[s:s + rb], d2[s:s + rb])
                _, up = raft(a, b, iters=20, test_mode=True)
                if host_io:
                    flows_host[s:s + rb].copy_(up, non_blocking=True)
            for _ in range(npairs):
                a, b = (hfl.to(dev, non_blocking=True), hmk.to(dev, non_blocking=True)) if host_io else (dfl, dmk)
                res = lafc(a, b, None)
                if host_io:
                    res[0].cpu()
            if host_io:
                torch.cuda.current_stream().synchronize()

        sampler.start()
        l0 = lib.COUNTERS["launches"]
        ms = parallel.max_over_ranks(_events(lambda: step(False), args.steps, args.warmup, flush, barrier), dev)
        launches = (lib.COUNTERS["launches"] - l0) // (args.steps + args.warmup)
        ms_e2e = parallel.max_over_ranks(_events(lambda: step(True), max(2, args.steps // 2), 2, flush, barrier), dev)
        clocks = sampler.stop()
        raft.enable_cuda_graph(False)
        lafc.net.enable_cuda_graph(False)
        with torch.no_grad():
            raft(d1[:rb], d2[:rb], iters=20, test_mode=True)
            lafc(dfl, dmk, None)
            lib.profile_start()
            raft(d1[:rb], d2[:rb], iters=20, test_mode=True)
            for _ in range(rb):
                lafc(dfl, dmk, None)
            roof, kernels = _dominant(lib.profile_stop(), 1, peaks)
        frames = T * world
        h2d = (h1.numel() + h2.numel()) * 4 + npairs * (hfl.numel() + hmk.numel()) * 4
        d2h = flows_host.numel() * 4 + npairs * 2 * (H // 2) * (W // 2) * 4
        scaling = "weak"
        par = f"pair-dp{world}"
        extra = {"raft_pairs_per_step": npairs, "lafc_calls_per_step": npairs, "raft_batch": rb,
                 "breakdown_note": "kernels/roofline from one instrumented eager batch of 4 RAFT pairs + 4 LAFC calls"}
    else:
        from fgt_b200.fgt_model import Model
        T, H, W = spec["T"], spec["H"], spec["W"]
        cfg = dict(synth.CFG_A)
        model = Model(cfg)
        model.load_state_dict(synth.make_state_dict(synth.fgt_param_shapes(cfg), seed=1, regime="scaled"))
        model = model.to(dev)
        model.net.enable_cuda_graph(True)
        sched = parallel.window_schedule(T)
        sizes = [len(nb) + len(ref) for _, nb, ref in sched]
        mine = parallel.shard_items(len(sched), rank, world, costs=sizes)
        clip = synth.fgt_inputs(seed=3, t=T, H=H, W=W)
        wins = [sched[i][1] + sched[i][2] for i in mine]
        # the rank's input = the frames its windows read (pinned, prepared once); like the reference driver
        # (tool/video_inpainting.py:445-470: the clip lives on the device, windows are index selections of it), the
        # end-to-end step uploads those frames ONCE per clip and gathers each window on the device
        need = sorted(set().union(*[set(w) for w in wins]))
        pos = {f: i for i, f in enumerate(need)}
        host = [t[:, need].contiguous().pin_memory() for t in clip]
        devin = [t.to(dev) for t in host]
        wins_l = [torch.tensor([pos[f] for f in w], device=dev) for w in wins]
        out_host = torch.empty(max(sizes), 3, H, W).pin_memory()

        def step(host_io):
            src = [h.to(dev, non_blocking=True) for h in host] if host_io else devin
            for ids, sel in zip(wins, wins_l):
                part = [t.index_select(1, sel) for t in src]
                o = model(*part)
                if host_io:
                    out_host[:len(ids)].copy_(o, non_blocking=True)
            if host_io:
                torch.cuda.current_stream().synchronize()

        sampler.start()
        l0 = lib.COUNTERS["launches"]
        ms = parallel.max_over_ranks(_events(lambda: step(False), args.steps, args.warmup, flush, barrier), dev)
        launches = (lib.COUNTERS["launches"] - l0) // (args.steps + args.warmup)
        ms_e2e = parallel.max_over_ranks(_events(lambda: step(True), max(2, args.steps // 2), 1, flush, barrier), dev)
        clocks = sampler.stop()
        model.net.enable_cuda_graph(False)
        ids = wins[0]
        part = [t.index_select(1, wins_l[0]) for t in devin]
        with torch.no_grad():
            model(*part)
            lib.profile_start()
            model(*part)
            roof, kernels = _dominant(lib.profile_stop(), 1, peaks)
        frames = T
        h2d = sum(h.numel() for h in host) * 4
        d2h = sum(len(w) for w in wins) * 3 * H * W * 4
        scaling = "strong"
        par = f"window-dp{world}"
        extra = {"windows": len(sched), "window_sizes": sizes, "windows_of_rank0": mine,
                 "peak_mem_gb": round(torch.cuda.max_memory_allocated() / 2 ** 30, 2),
                 "breakdown_note": f"kernels/roofline from one instrumented eager forward of a t={len(ids)} window"}
    if rank == 0:
        print(json.dumps({
            "kernels": kernels, "detail": extra,
            "metric": spec["metric"], "value": frames / (ms * 1e-3), "unit": "frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": scaling,
            "vs_baseline": None, "dtype": "bf16x3 (split-bf16 operands, fp32 accumulate)", "data": "synthetic",
            "config": {"workload": spec["workload"], "parallelism": par},
            "e2e": {"value": frames / (ms_e2e * 1e-3), "unit": "frames/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e,
                    "api": "pinned host inputs copied in and results copied out inside the timed region, one stream"
                           + ("" if args.config == 3 else "; the rank's frames are uploaded once per clip, windows gathered on the device")},
            "gpu_launches": launches, "clocks": clocks, "roofline": roof, "cpu_baseline": None, "impl": "fgt_b200",
        }), file=out, flush=True)
    if world > 1:
        dist.destroy_process_group()
