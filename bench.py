#!/usr/bin/env python
"""bench.py — inpainted frames/sec of FGT full inference at 432x240, T=10 (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl fgt_b200|reference|reference-gpu] [--config 2|3|4|5]
                    [--dump-outputs DIR]

Default (--config 2): a step is one Model.forward over one synthetic masked clip [1,10,3,240,432] (+flows,
masks) with seeded random weights of the reference architecture. `value` is measured with the inputs already
in HBM; `e2e` goes through the public API from pinned HOST buffers (H2D of the clip and D2H of the
inpainted frames inside the timed region). N>1: one process per GPU, each rank inpaints its own
clip window (the driver's window loop, tool/video_inpainting.py:710, is embarrassingly parallel:
no data-path collective), weak scaling, time = max over ranks. Additionally, at every N>1, ONE window is
split by frames over the ranks (FGT.enable_frame_sharding: the partitioning BASELINE.json's north_star names;
exchange per temporal layer) and reported as strong scaling under `frame_sharded` (and, compactly, in
`e2e.frame_sharded`, which the driver's record keeps).

--dump-outputs DIR (default config and impl): after the timed steps, rank 0 writes the inpainted frames that the last
timed step's Model.forward returned, [T,3,240,432] float32, to DIR/inpainted_frames.npy. Inputs and weights are seeded,
so two builds run with the same arguments can be compared output for output.

The other BASELINE configurations are separate lines: --config 3 (RAFT + LAFC at 480x864, T=20),
--config 4 (432x240 T=80 clip = 16 windows of the driver's schedule, windows sharded over the ranks),
--config 5 (1280x720 T=40 clip = 8 windows).

--impl reference times the CPU oracle port of the reference path (oracle/fgt_oracle.py, validated against the
unmodified reference in tests/golden) on the host cores — the reference itself is Python under
/root/reference and does not exist on the GPU box. --impl reference-gpu (and the `gpu_eager_baseline` key of
the default line) runs the same PyTorch restatement eagerly on the B200 (cuBLAS / cuDNN): the bar SURVEY.md
§2.2 names.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from fgt_b200 import synth  # noqa: E402

T, H, W = 10, 240, 432
RESULT_OUT = sys.stdout
METRIC = "inpainted_frames_per_sec_432x240_T10"
WORKLOAD = "FGT full inference (Model.forward), synthetic 432x240 clip T=10, random mask, seeded random weights"
CPU_THREADS_CAP = 32  # deterministic thread rule for the CPU arm: min(32, host cores); ATen slows down when oversubscribed


def config_dict(world):
    """Identical for every arm of config 2 (the driver compares the arms' config dicts)."""
    return {"workload": WORKLOAD, "frames_per_step_per_gpu": T, "parallelism": f"window-dp{world}"}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as fh:
            d = json.load(fh)
        return dict(hbm_gbs=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d["bf16_tflops_sustained"],
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def build_model(dev):
    from fgt_b200.fgt_model import Model
    cfg = dict(synth.CFG_A)
    sd = synth.make_state_dict(synth.fgt_param_shapes(cfg), seed=1, regime="scaled")
    m = Model(cfg)
    m.load_state_dict(sd)
    return m.to(dev), sd


def cpu_threads():
    n = min(CPU_THREADS_CAP, os.cpu_count() or 1)
    torch.set_num_threads(n)
    return n


def oracle_cpu(sd, clip, runs, warm=1):
    """frames/sec of the CPU oracle port on `clip`; returns (fps, mean seconds per forward, threads)."""
    from oracle import fgt_oracle as O
    sdn = O.strip_net(sd)
    threads = cpu_threads()
    times = []
    with torch.no_grad():
        for i in range(warm + runs):
            t0 = time.perf_counter()
            O.fgt_forward(sdn, *clip)
            if i >= warm:
                times.append(time.perf_counter() - t0)
    sec = sum(times) / len(times)
    return clip[0].shape[1] / sec, sec, threads


def oracle_gpu_eager(sd, clip, dev, runs=5, warm=2):
    """The same PyTorch restatement run eagerly on the GPU (cuBLAS / cuDNN kernels), fp32 with TF32 off and on."""
    from oracle import fgt_oracle as O
    sdn = {k: v.to(dev) for k, v in O.strip_net(sd).items()}
    dclip = [t.to(dev) for t in clip]
    out = {}
    old = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32, torch.backends.cudnn.benchmark)
    torch.backends.cudnn.benchmark = True
    try:
        for name, tf32 in (("fp32", False), ("tf32", True)):
            torch.backends.cuda.matmul.allow_tf32 = tf32
            torch.backends.cudnn.allow_tf32 = tf32
            ms = []
            with torch.no_grad():
                for i in range(warm + runs):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    O.fgt_forward(sdn, *dclip)
                    e1.record()
                    torch.cuda.synchronize()
                    if i >= warm:
                        ms.append(e0.elapsed_time(e1))
            m = sum(ms) / len(ms)
            out[name] = {"value": clip[0].shape[1] / (m * 1e-3), "unit": "frames/s", "ms_per_step": m}
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32, torch.backends.cudnn.benchmark = old
    out["how"] = (f"oracle/fgt_oracle.fgt_forward on CUDA tensors (PyTorch eager, cuBLAS/cuDNN, cudnn.benchmark), same clip "
                  f"and weights, {warm} warm-ups + {runs} CUDA-event-timed forwards, inputs resident on the device")
    return out


def run_reference(args, rank, world):
    """CPU arm: the oracle port of the reference path on the host cores (rank 0 only)."""
    if rank != 0:
        return
    cfg = dict(synth.CFG_A)
    sd = synth.make_state_dict(synth.fgt_param_shapes(cfg), seed=1, regime="scaled")
    from oracle import fgt_oracle as O
    sdn = O.strip_net(sd)
    threads = cpu_threads()
    # bounded sample: shrink the clip length only if K+W forwards of T=10 would exceed ~4 minutes
    probe = synth.fgt_inputs(seed=3, t=2, H=H, W=W)
    with torch.no_grad():
        O.fgt_forward(sdn, *probe)
        t0 = time.perf_counter()
        O.fgt_forward(sdn, *probe)
        per_frame = (time.perf_counter() - t0) / 2
    ts = T
    while ts > 2 and per_frame * ts * (args.steps + args.warmup) > 240.0:
        ts -= 2
    clip = synth.fgt_inputs(seed=3, t=ts, H=H, W=W)
    times = []
    with torch.no_grad():
        for i in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            O.fgt_forward(sdn, *clip)
            if i >= args.warmup:
                times.append(time.perf_counter() - t0)
    ms = 1e3 * sum(times) / len(times)
    fps = ts / (ms / 1e3)
    sample = f"{args.steps} forwards of a T={ts} 432x240 clip"
    if ts != T:
        sample += f" (T reduced from {T} only to bound the run time; frames/s is per frame)"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config_dict(args.gpus),
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "host_cores": os.cpu_count(), "kind": "port",
                         "sample": sample, "thread_rule": f"min({CPU_THREADS_CAP}, host cores)"},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }), file=RESULT_OUT, flush=True)


def run_reference_gpu(args, rank, world):
    """GPU-eager arm: the PyTorch restatement on the B200 through cuBLAS / cuDNN (rank 0 only)."""
    if rank != 0:
        return
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    cfg = dict(synth.CFG_A)
    sd = synth.make_state_dict(synth.fgt_param_shapes(cfg), seed=1, regime="scaled")
    clip = synth.fgt_inputs(seed=3, t=T, H=H, W=W)
    r = oracle_gpu_eager(sd, clip, dev, runs=args.steps, warm=args.warmup)
    print(json.dumps({
        "impl": "reference-gpu", "metric": METRIC, "value": r["fp32"]["value"], "unit": "frames/s", "n_gpus": 1,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["fp32"]["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32 (TF32 off); tf32 variant under gpu_eager_baseline",
        "data": "synthetic", "config": config_dict(1), "gpu_eager_baseline": r, "gpu_launches": 0,
    }), file=RESULT_OUT, flush=True)


# ----------------------------------------------------------------------------------------------------------
# algorithmic work of the three transformer modules (SURVEY.md §8d), per layer
# ----------------------------------------------------------------------------------------------------------
def module_flops(t, n=720, d=512, df=256, heads=4, zones=4, P=960, G=60, nwin=15, hidden=1960):
    tm = 4 * 2 * d * d * (t * n) + zones * heads * 4 * (t * n / zones) ** 2 * (d // heads)
    sw = t * (2 * (d + df) * df * P + 2 * (d + df) * d * (2 * P + G) + 2 * d * d * (P + G)
              + nwin * heads * 4 * 64 * (64 + G) * (d // heads) + 2 * d * d * n)
    ff = 2 * 2 * d * hidden * (t * n)
    return {"tmhsa": tm, "swmhsa": sw, "ffn": ff}


def aggregate(recs, reps, peaks):
    """Per-kernel and per-module sums of the per-launch CUDA-event times of `reps` instrumented eager forwards."""
    agg, mods = {}, {}
    for kern, tag, fl, by, ms, sc in recs:
        key = kern if kern != "flash" else ("flash_temporal" if tag.startswith("t") else "flash_spatial")
        a = agg.setdefault(key, dict(ms=0.0, flops=0.0, bytes=0.0, n=0))
        a["ms"] += ms / reps
        a["flops"] += fl / reps
        a["bytes"] += by / reps
        a["n"] += 1 / reps
        m = mods.setdefault(sc or "other", dict(ms=0.0, n=0))
        m["ms"] += ms / reps
        m["n"] += 1 / reps
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
    return agg, kernels, mods


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="fgt_b200", choices=["fgt_b200", "reference", "reference-gpu"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's output as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.config != 2 or args.impl != "fgt_b200"):
        ap.error("--dump-outputs is supported for the default --config 2 --impl fgt_b200 only")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    # stdout carries exactly one JSON line: anything native libraries print to fd 1 (e.g. NCCL's version banner)
    # is sent to stderr, and the result line goes to the saved descriptor
    global RESULT_OUT
    sys.stdout.flush()
    RESULT_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.config != 2:
        from tools import bench_other
        return bench_other.run(args, rank, local_rank, world, RESULT_OUT)
    if args.impl == "reference":
        return run_reference(args, rank, world)
    if args.impl == "reference-gpu":
        return run_reference_gpu(args, rank, world)
    assert args.warmup >= 3, "timing rules: at least 3 warm-up steps"
    import torch.distributed as dist
    from fgt_b200 import lib, parallel
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=dev)
    model, sd = build_model(dev)
    use_graph = os.environ.get("FGT_BENCH_GRAPH", "1") != "0"   # 0: eager launches (fixed kernel count per step, for ncu)
    model.net.enable_cuda_graph(use_graph)  # public option: whole forward replayed as one CUDA graph per geometry
    clip = synth.fgt_inputs(seed=3 + rank, t=T, H=H, W=W)
    host = [t.contiguous().pin_memory() for t in clip]
    devin = [t.to(dev) for t in host]
    out_host = torch.empty(T, 3, H, W).pin_memory()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(step_fn, steps=None, warmup=None):
        """W warm-ups then K steps; per-step CUDA events on the launching stream, L2 flushed (untimed)
        between steps; returns (mean ms/step over ranks' max, launches per step)."""
        steps = args.steps if steps is None else steps
        warmup = args.warmup if warmup is None else warmup
        with torch.no_grad():
            for _ in range(warmup):
                step_fn()
            barrier()
            evs = []
            l0 = lib.COUNTERS["launches"]
            for _ in range(steps):
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                step_fn()
                e1.record()
                evs.append((e0, e1))
            barrier()
            launches = lib.COUNTERS["launches"] - l0
        total_ms = sum(a.elapsed_time(b) for a, b in evs)
        return parallel.max_over_ranks(total_ms, dev) / steps, launches

    last = {}

    def step_device():
        last["out"] = model(*devin)   # kept for --dump-outputs: each step replaces the previous step's output

    def step_e2e():
        d = [h.to(dev, non_blocking=True) for h in host]
        out_host.copy_(model(*d), non_blocking=True)
        torch.cuda.current_stream().synchronize()

    def timed_streamed():
        """e2e through fgt_b200.streaming.ClipStreamer: K host-resident clips in, K host-resident results out;
        every clip's H2D and every result's D2H happen inside the timed region, overlapped with the
        neighbouring clips' forwards on separate streams. One event pair around the whole K-step region."""
        from fgt_b200.streaming import ClipStreamer
        st = ClipStreamer(model, host, dev)
        for _ in st.run([host] * args.warmup):
            pass
        barrier()
        cur = torch.cuda.current_stream(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(cur)
        n_out = 0
        for o in st.run([host] * args.steps):
            n_out += 1
        cur.wait_stream(st.s_out)
        e1.record(cur)
        barrier()
        assert n_out == args.steps
        return parallel.max_over_ranks(e0.elapsed_time(e1), dev) / args.steps, st

    def timed_frame_sharded(tw, fh=H, fw=W, steps=10):
        """N>1: ONE tw-frame window sharded by frames over the ranks (FGT.enable_frame_sharding: P2P exchange fused
        into the LayerNorm kernel vs NCCL all-gather) — strong scaling of a single forward; the one-GPU time of
        the same window is measured in the same run (every rank runs it; max over ranks)."""
        mine = parallel.shard_items(tw, rank, world)
        clip0 = synth.fgt_inputs(seed=3, t=tw, H=fh, W=fw)    # every rank: the same window, its own frames
        full = [t.to(dev) for t in clip0]
        model.net.enable_frame_sharding(None)
        model.net.enable_cuda_graph(True)
        ms1, _ = timed(lambda: model(*full), steps=steps, warmup=3)
        del full
        model.net._drop_graphs()                               # (the captured graph holds the workspaces' addresses)
        model.net._geo.clear()                                 # drop the full window's workspaces (30+ GB at 720p)
        torch.cuda.empty_cache()
        res = {"frames": tw, "size": f"{fw}x{fh}", "ms_one_gpu": ms1, "frames_per_rank": parallel.frame_counts(tw, world)}
        if not mine:
            return res
        part = [t[:, mine[0]:mine[-1] + 1].contiguous().to(dev) for t in clip0]
        for exchange in ("p2p", "nccl"):
            model.net.enable_frame_sharding(tw, exchange=exchange)
            model.net.enable_cuda_graph(exchange == "p2p")   # kernels only -> replayable; NCCL calls stay eager
            try:
                res["ms_" + exchange], _ = timed(lambda: model(*part), steps=steps, warmup=3)
            finally:
                model.net.enable_cuda_graph(False)
                model.net.enable_frame_sharding(None)
        best = min(res["ms_p2p"], res["ms_nccl"])
        res.update(value=tw / (best * 1e-3), unit="frames/s", speedup=ms1 / best, efficiency=ms1 / best / world,
                   scaling="strong")
        return res

    def timed_driver_schedule():
        """SURVEY 8d: the driver's own window schedule for a 10-frame clip (tool/video_inpainting.py:709-717 with
        step 10, stride 5): f=0 -> 6 frames, f=5 -> all 10; frames/s = 10 emitted frames / (t6 + t10). Device-resident
        inputs, same event timing as `value`."""
        sched = parallel.window_schedule(T)
        ms = []
        for _, nb, ref in sched:
            ids = nb + ref
            part = [t[:, ids].contiguous() for t in devin]
            m, _ = timed(lambda: model(*part), steps=10, warmup=3)
            ms.append(m)
        return {"windows_t": [len(nb) + len(ref) for _, nb, ref in sched], "ms_per_window": ms,
                "value": T * world / (sum(ms) * 1e-3), "unit": "frames/s",
                "note": "10 output frames per clip / time of the clip's two windows (6 + 10 input frames)"}

    sampler = ClockSampler(local_rank)
    sampler.start()
    ms_dev, launches = timed(step_device)
    if args.dump_outputs and rank == 0:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "inpainted_frames.npy"), last["out"].float().cpu().numpy())
    last.clear()
    ms_e2e_serial, _ = timed(step_e2e)
    ms_e2e, streamer = timed_streamed()
    clocks = sampler.stop()
    driver_sched = None
    try:
        driver_sched = timed_driver_schedule()
    except Exception as exc:  # noqa: BLE001 - an extra line, never fatal for the main measurement
        print(f"[bench] driver-schedule measurement failed: {exc}", file=sys.stderr)

    # per-kernel / per-module breakdown: CUDA events around every launch of 3 more forwards (not part of `value`)
    peaks = load_peaks()
    model.net.enable_cuda_graph(False)  # per-launch CUDA events need the eager launch sequence
    reps = 3
    with torch.no_grad():
        model(*devin)
        lib.profile_start()
        for _ in range(reps):
            model(*devin)
    agg, kernels, mods = aggregate(lib.profile_stop(), reps, peaks)
    mf = module_flops(T)
    layers = {"tmhsa": 4, "swmhsa": 4, "ffn": 8}
    modules = {}
    for name, m in sorted(mods.items(), key=lambda kv: -kv[1]["ms"]):
        e = {"ms_per_step": round(m["ms"], 4), "launches_per_step": round(m["n"])}
        if name in mf:
            per_layer_us = m["ms"] * 1e3 / layers[name]
            tf = mf[name] / (per_layer_us * 1e-6) / 1e12
            e.update(layers=layers[name], us_per_layer=round(per_layer_us, 1), gflop_per_layer=round(mf[name] / 1e9, 2),
                     achieved_tflops=round(tf, 1), frac=round(tf / peaks["tf_sustained"], 4))
        modules[name] = e
    worst = min((k for k in modules if "frac" in modules[k]), key=lambda k: modules[k]["frac"], default=None)
    dk, da = max(agg.items(), key=lambda kv: kv[1]["ms"])
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as fh:
            traffic = json.load(fh).get(dk)
    if da["flops"] > 0:
        ach = da["flops"] / (da["ms"] * 1e-3) / 1e12
        roof = {"kernel": dk, "bound": "tensor", "achieved": ach, "peak": peaks["tf_sustained"], "unit": "TFLOP/s",
                "frac": ach / peaks["tf_sustained"], "traffic": traffic, "peak_source": peaks["source"] + ", sustained bf16",
                "note": "algorithmic FLOPs; split-bf16 layers execute 3 MMAs per algorithmic one (ceiling 1/3), the "
                        "flow branch 1 (see dtype)"}
    else:
        ach = da["bytes"] / (da["ms"] * 1e-3) / 1e9
        roof = {"kernel": dk, "bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": ach / peaks["hbm_gbs"], "traffic": traffic, "peak_source": peaks["source"]}
    roof["modules"] = {k: {kk: v[kk] for kk in ("us_per_layer", "gflop_per_layer", "achieved_tflops", "frac")}
                       for k, v in modules.items() if "frac" in v}
    roof["worst_module"] = worst
    roof["modules_how"] = ("per layer: sum of the CUDA-event times of the module's launches in 3 instrumented eager "
                           "forwards / SURVEY 8d algorithmic FLOPs / sustained bf16 peak")

    eager = None
    if rank == 0 and world == 1 and not args.no_eager_baseline:
        try:
            eager = oracle_gpu_eager(sd, clip, dev)
        except Exception as exc:  # noqa: BLE001
            print(f"[bench] GPU-eager baseline failed: {exc}", file=sys.stderr)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        fps_cpu, sec, threads = oracle_cpu(sd, clip, runs=3)
        cpu = {"value": fps_cpu, "unit": "frames/s", "cores": threads, "host_cores": os.cpu_count(), "kind": "port",
               "thread_rule": f"min({CPU_THREADS_CAP}, host cores)",
               "sample": f"1 warm-up + 3 forwards of the same T=10 432x240 clip ({sec:.2f} s each), oracle/fgt_oracle.py"}

    fshard = None
    if world > 1 and os.environ.get("FGT_BENCH_FRAME_SHARD", "1") != "0":
        fshard = {}
        for tw in (10, 16, 18):
            if world > tw:
                continue
            try:
                fshard[f"T{tw}"] = timed_frame_sharded(tw)
            except Exception as exc:  # noqa: BLE001 - reported, never fatal for the main line
                print(f"[bench] frame-sharded measurement (T={tw}) failed: {exc}", file=sys.stderr)
                fshard[f"T{tw}"] = {"error": str(exc)[:200]}
        # BASELINE config 5's shape (1280x720, window-partition + global-token path, 21-26 k-key temporal zones): where a
        # rank's share of a window is heavy enough for frame sharding to pay at 8 GPUs
        if os.environ.get("FGT_BENCH_FS_720P", "1") != "0" and world <= 16:
            try:
                fshard["T16_1280x720"] = timed_frame_sharded(16, 720, 1280, steps=5)
            except Exception as exc:  # noqa: BLE001
                print(f"[bench] frame-sharded measurement (720p) failed: {exc}", file=sys.stderr)
                fshard["T16_1280x720"] = {"error": str(exc)[:200]}
            finally:
                model.net._geo.clear()
                torch.cuda.empty_cache()
    if rank == 0:
        frames = T * world
        h2d = sum(t.numel() * t.element_size() for t in host)
        d2h = out_host.numel() * out_host.element_size()
        fs_compact = None
        if fshard:
            fs_compact = {k: {kk: (round(v[kk], 4) if isinstance(v[kk], float) else v[kk])
                              for kk in ("ms_one_gpu", "ms_p2p", "ms_nccl", "speedup", "efficiency") if kk in v}
                          for k, v in fshard.items()}
        # bulky detail first, the contract's keys last (a truncated tail of the line keeps the headline)
        print(json.dumps({
            "kernels": kernels, "modules": modules, "driver_schedule": driver_sched, "frame_sharded": fshard,
            "timing": {"cuda_graph": use_graph,
                       "l2": "256 MiB buffer rewritten between steps (untimed); activations (>1 GB) exceed L2"},
            "metric": METRIC, "value": frames / (ms_dev * 1e-3), "unit": "frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16x3 (split-bf16 operands, 3 MMAs, fp32 accumulate); flow branch (flow encoder, f_patch2vec, "
                     "flow gate) bf16x1",
            "data": "synthetic", "config": config_dict(world),
            "e2e": {"value": frames / (ms_e2e * 1e-3), "unit": "frames/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e,
                    "api": "fgt_b200.streaming.ClipStreamer(Model).run(pinned host clips) -> pinned host frames; "
                           "H2D / forward / D2H of neighbouring clips overlap on three streams; one event pair "
                           "around all K steps, inputs re-read from host every step",
                    "serial_value": frames / (ms_e2e_serial * 1e-3), "serial_ms_per_step": ms_e2e_serial,
                    "serial_api": "x.to(device) -> Model.forward -> out.cpu(), one stream, per-step events",
                    "frame_sharded": fs_compact},
            "gpu_launches": launches, "clocks": clocks, "roofline": roof,
            "gpu_eager_baseline": eager, "cpu_baseline": cpu, "impl": "fgt_b200",
        }), file=RESULT_OUT, flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
