#!/usr/bin/env python
"""bench.py -- frames/s end-to-end (conv + PAF parse), OpenPose-COCO VGG-19 368x656, batch 16 per GPU.

    python bench.py --gpus 1 --steps 20 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the reference's own CPU parser (oracle/_ref) on the host cores

One "step" = one pass of the hot path over one batch of 16 synthetic frames per GPU (weak scaling:
frames shard across GPUs, SURVEY 8e): frame pre-processing + every conv of OpenPose-VGG19 (random-init
weights of the real architecture) + the PAF parse of the batch (+ for N>1 the NCCL gather of the
keypoint records to rank 0).  Because random weights give structureless heat-maps, seeded synthetic
crowd tensors are copied over the backbone's outputs after the last conv (hp_engine_set_output_override,
SURVEY 8d) -- all conv work is still executed; this is stated in config.parse_input.

  value : device-resident inputs (u8 frames already in HBM), results left on the device (rank 0 after gather);
          hp_pose_submit_u8_device / hp_pose_collect (CUDA-graph replay, two batches in flight)
  e2e   : the public host call hp_pose_submit_u8_host / hp_pose_collect -- pinned host frames H2D, human_t records D2H, every step
  roofline : the conv kernel (dominant): algorithmic FLOPs / CUDA-event time of the conv launches, measured in
             the timed region on the launching stream, vs the measured cuBLAS bf16 peak
  cpu_baseline : the reference's CPU parser timed on this host (parse stage only: the reference never runs
             the convs on a CPU; its engine is TensorRT)
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# workloads (BASELINE.json configs).  The default -- and the only one the headline metric is quoted on -- is cfg3.
WORKLOADS = {
    "cfg3": dict(name="cfg3: OpenPose-COCO VGG-19 368x656, batch 16 per GPU, frame-sharded", graph="openpose_vgg19", in_h=368, in_w=656,
                 batch=16, persons=(10, 20), algo_flops=484.6e9, arch="OpenPose-VGG19 (6 stages), 484.6 GFLOP/frame"),
    "cfg2": dict(name="cfg2: Lightweight-OpenPose (MobilenetThin) 368x432, batch 8", graph="mobilenet_thin_openpose", in_h=368, in_w=432,
                 batch=8, persons=(1, 5), algo_flops=22.3e9, arch="MobilenetThin-OpenPose (6 stages), 22.3 GFLOP/frame"),
    "cfg4": dict(name="cfg4: OpenPose-ResNet50 (LW-OpenPose head, stride 8) 368x432, batch 32 per GPU, synthetic crowd", graph="resnet50_lw_openpose",
                 in_h=368, in_w=432, batch=32, persons=(10, 20), algo_flops=136.7e9, arch="ResNet50 + LW-OpenPose head, 136.7 GFLOP/frame"),
    "cfg5": dict(name="cfg5: OpenPifPaf ResNet50 385x385, batch 16 (pif/paf field decode)", graph="resnet50_pifpaf", in_h=385, in_w=385,
                 batch=16, persons=(2, 8), algo_flops=100.2e9, arch="ResNet50 (stride 16, no max-pool) + PIF/PAF heads, 100.2 GFLOP/frame", pifpaf=True),
}
IN_H, IN_W, HF, WF, BATCH, PERSONS, ALGO_FLOPS_PER_FRAME = 368, 656, 46, 82, 16, (10, 20), 484.6e9
WL = WORKLOADS["cfg3"]
N_INPUT_SETS = 12                    # distinct input batches rotated so that the frames alone exceed the 126 MB L2


def select_workload(key):
    global IN_H, IN_W, HF, WF, BATCH, PERSONS, ALGO_FLOPS_PER_FRAME, WL
    WL = WORKLOADS[key]
    IN_H, IN_W, BATCH, PERSONS, ALGO_FLOPS_PER_FRAME = WL["in_h"], WL["in_w"], WL["batch"], WL["persons"], WL["algo_flops"]
    HF, WF = IN_H // 8, IN_W // 8
    if WL.get("pifpaf"):
        HF, WF = (IN_H - 1) // 8 + 1, (IN_W - 1) // 8 + 1     # 49 x 49 fields for 385 x 385


def METRIC():
    return "frames/sec end-to-end (conv+PAF parse) OpenPose-COCO 368x656" if WL is WORKLOADS["cfg3"] else f"frames/sec end-to-end (conv+PAF parse) {WL['name']}"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return d, "measured"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """samples nvidia-smi during the timed region (B200_PROFILING.md clocks line)"""

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def crowd_tensors(seed: int):
    from hyperpose_b200 import synthetic as syn
    return syn.make_batch_tensors(seed, BATCH, PERSONS, HF, WF)


# ------------------------------------------------------------------------------------------------
# CPU baseline: the reference's own src/paf.cpp (oracle/_ref) or the oracle port, parse stage only
# ------------------------------------------------------------------------------------------------
def cpu_parse_rate(conf, paf, seconds: float, threads: int):
    """frames/s of the CPU parser on the host cores; one parser replica per thread, frames round-robin
    (the reference's stream API does exactly this: stream.hpp:139,365-373)."""
    import oracle
    kind = "reference" if oracle.ref_available() else "port"
    n = conf.shape[0]
    counts = [0] * threads
    stop = time.time() + seconds

    def work(t):
        if kind == "reference":
            rp = oracle.RefParser()
            fn = lambda i: rp.process(conf[i], paf[i])
        else:
            fn = lambda i: oracle.oracle_process(conf[i], paf[i])
        i = t
        fn(i % n)  # first call allocates (paf.cpp:321-332): not timed
        t0 = time.time()
        while time.time() < stop:
            fn(i % n)
            i += threads
            counts[t] += 1
        return time.time() - t0

    t_start = time.time()
    ths = [threading.Thread(target=work, args=(t,)) for t in range(threads)]
    for th in ths:
        th.start()
    for th in ths:
        th.join()
    wall = time.time() - t_start
    return sum(counts) / max(wall, 1e-9), kind


def cpu_threads():
    """every host thread this process may use (affinity mask AND cgroup CPU quota), independent of OMP_NUM_THREADS (torchrun
    sets it to 1)"""
    try:
        n = max(1, len(os.sched_getaffinity(0)))
    except Exception:
        n = os.cpu_count() or 1
    try:    # cgroup v2 quota: "<quota> <period>" or "max <period>"
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            n = max(1, min(n, int(float(q) / float(per) + 0.5)))
    except Exception:
        pass
    return n


def cpu_conv_threads():
    """thread count for the conv stage of the CPU arm: one per PHYSICAL core the process may use.  (An OpenMP team wider than
    the cores it can actually run on collapses at every barrier: measured on a 128-thread host, 128 threads -> 26 s per frame
    against 0.9 s with 64.)"""
    n = cpu_threads()
    try:
        import psutil
        phys = psutil.cpu_count(logical=False)
        if phys:
            n = max(1, min(n, phys))
    except Exception:
        n = max(1, n // 2) if n >= 16 else n
    return n


_CONV_THREADS = {}


def calibrate_conv_threads(graph_name: str):
    """picks the conv-stage thread count by measurement: the graph on ONE quarter-area frame with the physical-core count and with
    half of it (SMT siblings / cgroup quotas make "all threads" the slow choice on some hosts); cached per graph."""
    if graph_name in _CONV_THREADS:
        return _CONV_THREADS[graph_name]
    import torch
    from hyperpose_b200 import models, synthetic as syn
    from oracle import torch_backbone
    n = cpu_conv_threads()
    cands = sorted({n, max(1, n // 2)}, reverse=True)
    best, best_t = cands[-1], None
    if len(cands) > 1:
        graph = getattr(models, graph_name)(seed=0)
        probe = syn.make_frames_u8(3, 1, (IN_H // 16) * 8, (IN_W // 16) * 8)
        for c in cands:
            torch.set_num_threads(c)
            with torch.no_grad():
                torch_backbone.run_graph(graph, probe, device="cpu")     # warm-up (primitive caches)
                t0 = time.time()
                torch_backbone.run_graph(graph, probe, device="cpu")
                dt = time.time() - t0
            if best_t is None or dt < best_t:
                best, best_t = c, dt
    _CONV_THREADS[graph_name] = best
    return best


def cpu_conv_port(graph_name: str, n_frames: int):
    """conv stage on the host cores: oracle/torch_backbone.py (plain PyTorch fp32) on a batch of `n_frames` synthetic frames with an
    EXPLICIT, measured thread count (torch.set_num_threads: torchrun's OMP_NUM_THREADS=1 does not apply; calibrate_conv_threads).
    The reference has no CPU implementation of its convs (TensorRT on a GPU, src/tensorrt.cpp:387-396), so this stage
    of the CPU arm is a port, the parse stage is the reference's own code."""
    import torch
    from hyperpose_b200 import models, synthetic as syn
    from oracle import torch_backbone
    threads = calibrate_conv_threads(graph_name)
    torch.set_num_threads(threads)
    graph = getattr(models, graph_name)(seed=0)
    frames = syn.make_frames_u8(2, n_frames, IN_H, IN_W)

    def run():
        with torch.no_grad():
            torch_backbone.run_graph(graph, frames, device="cpu")
    return run, torch.get_num_threads()


def cpu_parse_batch(conf, paf, n_frames, threads):
    """the reference's own parser over `n_frames` frames, one replica per thread (what its stream API does, stream.hpp:139,365-373);
    returns a callable that parses the batch once"""
    import oracle
    kind = "reference" if oracle.ref_available() else "port"
    threads = max(1, min(threads, n_frames))
    if kind == "reference":
        reps = [oracle.RefParser() for _ in range(threads)]
        fns = [lambda i, r=r: r.process(conf[i % conf.shape[0]], paf[i % paf.shape[0]]) for r in reps]
    else:
        fns = [lambda i: oracle.oracle_process(conf[i % conf.shape[0]], paf[i % paf.shape[0]]) for _ in range(threads)]

    def run():
        def work(t):
            for i in range(t, n_frames, threads):
                fns[t](i)
        ths = [threading.Thread(target=work, args=(t,)) for t in range(threads)]
        for th in ths:
            th.start()
        for th in ths:
            th.join()
    return run, kind, threads


def bench_config(world: int = 1):
    """the `config` object BOTH arms print (the driver compares them)"""
    pif = bool(WL.get("pifpaf"))
    return {"workload": WL["name"],
            "global_batch": world * BATCH, "input": f"u8 frames {IN_H}x{IN_W}x3, random (default_rng)",
            "weights": "random-init (He-normal, seed 0) of the reference architecture: " + WL["arch"],
            "parse_input": f"synthetic {'PIF/PAF fields' if pif else 'crowd tensors'} ({PERSONS[0]}-{PERSONS[1]} persons/frame) copied over the conv outputs after the last conv",
            "l2": f"{N_INPUT_SETS} distinct input batches rotated ({N_INPUT_SETS * BATCH * IN_H * IN_W * 3 / 1e6:.0f} MB > L2); activations (>1 GB/step) stream through",
            "parallelism": f"dp{world} (frames shard; NCCL all-gather of keypoint records only)" if world > 1 else "single GPU"}


def run_reference(args):
    """--impl reference: the path on this host's CPU cores, same metric / unit / config as the GPU arm (frames/s through conv + parse
    on batches of the workload's frames).  Parse stage = the reference's own src/paf.cpp compiled verbatim (oracle/_ref), one replica
    per thread like its stream API; conv stage = a PyTorch fp32 port of the same graph on ALL host threads (explicit
    torch.set_num_threads: the reference runs its convs in TensorRT on a GPU and has no CPU implementation of them, so no
    "reference" conv stage can exist on a CPU).  Each step is a bounded sample: as many frames of the batch as keep the whole
    --steps/--warmup run within ~3 minutes (the full batch of 16 when the host is fast enough); frames/s does not depend on it."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle
    oracle.build()
    conf, paf = crowd_tensors(1000)
    cores = cpu_threads()
    # calibrate: one frame through the conv stage
    probe, conv_threads = cpu_conv_port(WL["graph"], 1)
    probe()
    t0 = time.time(); probe(); t_frame = time.time() - t0
    budget_s = 170.0
    n_steps_total = max(args.warmup, 1) + args.steps
    frames_per_step = int(max(1, min(BATCH, budget_s / n_steps_total / max(t_frame, 1e-3))))
    conv_run, conv_threads = cpu_conv_port(WL["graph"], frames_per_step)
    parse_run, kind, parse_threads = cpu_parse_batch(conf, paf, frames_per_step, cores)
    t_conv = t_parse = 0.0

    def step(timed):
        nonlocal t_conv, t_parse
        t0 = time.time()
        conv_run()
        t1 = time.time()
        parse_run()
        t2 = time.time()
        if timed:
            t_conv += t1 - t0
            t_parse += t2 - t1

    for _ in range(max(args.warmup, 1)):
        step(False)
    t0 = time.time()
    for _ in range(args.steps):
        step(True)
    dt = time.time() - t0
    fps = args.steps * frames_per_step / dt
    # the parser alone with every host thread: the reference's own code on the stage it does run on a CPU
    parse_rate, _ = cpu_parse_rate(conf, paf, 3.0, min(cores, BATCH))
    cfg = bench_config(max(1, args.gpus))
    line = {
        "impl": "reference", "metric": METRIC(), "value": fps, "unit": "frames/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": max(conv_threads, parse_threads), "kind": "port",
                         "sample": f"{frames_per_step} of the batch's {BATCH} frames per step ({args.steps} steps): conv stage {t_conv / args.steps / frames_per_step * 1e3:.0f} ms/frame "
                                   f"(PyTorch fp32 port of the same graph, torch.set_num_threads({conv_threads}); the reference's convs are TensorRT-on-GPU, no CPU implementation exists) + "
                                   f"parse stage {t_parse / args.steps / frames_per_step * 1e3:.2f} ms/frame ({kind} parser src/paf.cpp, {parse_threads} replicas on threads) of {cores} usable host threads",
                         "frames_per_step": frames_per_step, "conv_threads": conv_threads, "parse_threads": parse_threads,
                         "parse_only": {"value": parse_rate, "unit": "frames/s", "cores": min(cores, BATCH), "kind": kind}},
        "parse_only": {"value": parse_rate, "unit": "frames/s", "cores": min(cores, BATCH), "kind": kind,
                       "what": "the reference's own CPU code for the stage it runs on a CPU (src/paf.cpp), same synthetic crowd tensors as the GPU arm's parse stage"},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def dump_humans(out_dir, prefix, humans, cap):
    """the human_t records a caller of the timed path receives for one batch (`humans`: one HUMAN_DT array per frame), as
    float32 arrays: <prefix>_human_parts.npy [N, cap, 18, 4] (has_value, x, y, score of every part), <prefix>_human_scores.npy
    [N, cap], both zero past a frame's count, and <prefix>_human_counts.npy [N].
    The timed path copies seeded synthetic conf / PAF tensors over the backbone's outputs (set_output_override), so these records
    depend on the parse stage alone: equal dumps from two builds say nothing about their conv kernels (tests/test_engine_gpu.py
    compares those with a PyTorch reference)."""
    os.makedirs(out_dir, exist_ok=True)
    parts = np.zeros((len(humans), cap, 18, 4), np.float32)
    scores = np.zeros((len(humans), cap), np.float32)
    for i, h in enumerate(humans):
        p = h["parts"]
        parts[i, :len(h)] = np.stack([p["has_value"], p["x"], p["y"], p["score"]], axis=-1)
        scores[i, :len(h)] = h["score"]
    np.save(os.path.join(out_dir, f"{prefix}_human_parts.npy"), parts)
    np.save(os.path.join(out_dir, f"{prefix}_human_scores.npy"), scores)
    np.save(os.path.join(out_dir, f"{prefix}_human_counts.npy"), np.array([len(h) for h in humans], np.float32))


# ------------------------------------------------------------------------------------------------
def measure(args, key, dist_ctx, headline=True):
    """one workload on this rank's GPU; returns (on rank 0) the JSON-line dict.  headline=False: the `extra_configs` entries
    (shorter pre-load, no CPU baseline, no parse-batch sweep)."""
    import torch
    import torch.distributed as dist
    from hyperpose_b200 import capi, models, synthetic as syn
    select_workload(key)
    rank, local_rank, world, dev = dist_ctx
    steps = args.steps
    warmup = args.warmup

    graph = getattr(models, WL["graph"])(seed=0)
    pack = graph.to_pack()
    engine = capi.Engine(pack, (IN_W, IN_H), max_batch_size=BATCH, device=local_rank, dtype=args.dtype)
    del pack
    PIFPAF = bool(WL.get("pifpaf"))
    HCAP = 128 if PIFPAF else 64
    if PIFPAF:
        parser = capi.PifPafParser(IN_H, IN_W, 0.1, device=local_rank)
    else:
        parser = capi.PafParser(0.05, 0.05, device=local_rank)
        parser.set_capacity(peaks_per_part=128, candidates_per_limb=2048, humans=HCAP)

    # inputs: N_INPUT_SETS distinct batches of frames (device + pinned host), one set of crowd tensors per rank
    rng_seed = 2 + 1000 * rank
    frames_host = [torch.from_numpy(syn.make_frames_u8(rng_seed + i, BATCH, IN_H, IN_W)).pin_memory() for i in range(N_INPUT_SETS)]
    frames_np = [f.numpy() for f in frames_host]
    frames_dev = [f.to(dev) for f in frames_host]
    if PIFPAF:
        fields = [syn.make_pifpaf_fields(1000 * (rank + 1) + i, PERSONS, HF, WF) for i in range(BATCH)]
        conf_np = np.stack([f[0] for f in fields]).reshape(BATCH, 85, HF, WF)
        paf_np = np.stack([f[1] for f in fields]).reshape(BATCH, 171, HF, WF)
    else:
        conf_np, paf_np = crowd_tensors(1000 + rank)
    d_conf = torch.from_numpy(conf_np).to(dev)
    d_paf = torch.from_numpy(paf_np).to(dev)
    engine.set_output_override(d_conf.data_ptr(), d_paf.data_ptr())
    out_conf_ptr, out_paf_ptr, _ = engine.device_outputs()

    # everything is enqueued on the ENGINE's own stream (events, timing, result copies): wrap it for torch
    st = torch.cuda.ExternalStream(engine.device_outputs()[2], device=dev)
    rec_bytes = capi.HUMAN_DT.itemsize
    # keypoint records + per-frame counts of one batch in ONE buffer (a single NCCL all-gather per step), double-buffered so
    # that the gather of batch i runs on a side stream while batch i+1 is computed
    hum_bytes = BATCH * HCAP * rec_bytes
    res_bufs = [torch.zeros(hum_bytes + BATCH * 4, dtype=torch.uint8, device=dev) for _ in range(2)]
    gath_bufs = [torch.zeros(world * (hum_bytes + BATCH * 4), dtype=torch.uint8, device=dev) for _ in range(2)] if world > 1 else None
    sg = torch.cuda.Stream(device=dev)
    ev_res = [torch.cuda.Event() for _ in range(2)]
    ev_gat = [torch.cuda.Event() for _ in range(2)]
    gstate = {"n": 0}
    use_gather = world > 1 and not PIFPAF and not os.environ.get("HPB_NO_GATHER")   # (diagnostic switch; the gather is part of the metric)

    def gather_results():
        if PIFPAF:
            return    # config 5 is a single-GPU config: records stay in the decoder's device buffer
        k = gstate["n"] & 1
        if gstate["n"] >= 2 and use_gather:
            st.wait_event(ev_gat[k])              # the gather that last read this buffer has finished
        buf = res_bufs[k]
        parser.copy_results_device(buf.data_ptr(), buf.data_ptr() + hum_bytes, BATCH, HCAP, st.cuda_stream)
        if use_gather:
            ev_res[k].record(st)
            sg.wait_event(ev_res[k])
            with torch.cuda.stream(sg):
                dist.all_gather_into_tensor(gath_bufs[k], buf)   # ~300 KB per rank, off the conv stream
            ev_gat[k].record(sg)
        gstate["n"] += 1

    def drain_gather():
        if use_gather:
            for k in range(2):
                if gstate["n"] > k:
                    st.wait_event(ev_gat[k])

    # value: frames already resident in HBM, results left on the device (rank 0 after the gather).  The launch sequence of a
    # batch is replayed from the CUDA graph hp_pose_submit_u8_device captured (two batches in flight: the host collects batch
    # i-1 while batch i runs); --no-graph (and the OpenPifPaf workload) launches every kernel on the stream instead.
    # (OpenPifPaf: the same two-deep submit / collect, without a CUDA graph -- the decoder runs on its own stream underneath the next
    #  batch's convolutions: hp_pose_submit_pifpaf_u8_device)
    use_graph = not args.no_graph
    dpend = {"t": None}
    pstate = {"events": None}     # pass B: CUDA events around the parser launches of every step

    def step_device(i):
        if use_graph:
            t = engine.submit_pose_device(parser, frames_dev[i % N_INPUT_SETS].data_ptr(), BATCH)
            gather_results()
            if dpend["t"] is not None:
                engine.collect_pose(dpend["t"], cap=HCAP)
            dpend["t"] = t
            return
        engine.infer_u8_device(frames_dev[i % N_INPUT_SETS].data_ptr(), BATCH, st.cuda_stream)
        pe = pstate["events"]
        if pe is not None:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(st)
        if PIFPAF:
            parser.process_device(out_conf_ptr, out_paf_ptr, BATCH, HF, WF, st.cuda_stream)
        else:
            parser.process_device(out_conf_ptr, out_paf_ptr, BATCH, 19, 38, HF, WF, st.cuda_stream)
        if pe is not None:
            b.record(st)
            pe.append((a, b))
        gather_results()

    def drain_device():
        if dpend["t"] is not None:
            h = engine.collect_pose(dpend["t"], cap=HCAP)
            dpend["t"] = None
            dpend["last"] = h
            return h

    # e2e: the public host call, pinned host frames in, human_t records out -- two batches in flight
    # (hp_pose_submit_u8_host / hp_pose_collect: H2D of batch i+1 under the convs of batch i, CUDA-graph replay)
    pend = {"t": None}

    def step_host(i):
        t = engine.submit_pose(parser, frames_np[i % N_INPUT_SETS])
        humans = engine.collect_pose(pend["t"], cap=HCAP) if pend["t"] is not None else None
        pend["t"] = t
        return humans

    def drain_host():
        if pend["t"] is not None:
            h = engine.collect_pose(pend["t"], cap=HCAP)
            pend["t"] = None
            return h

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n_steps, n_warm, profile=False):
        for i in range(n_warm):
            fn(i)
        if fn is step_host:
            drain_host()
        if fn is step_device:
            drain_device()
        barrier()
        l0 = engine.launch_count + parser.launch_count
        if profile:
            engine.set_profiling(True)
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(st)
        t0 = time.time()
        for i in range(n_steps):
            fn(n_warm + i)
        if fn is step_host:
            drain_host()
        if fn is step_device:
            drain_device()
        drain_gather()                                # the timed region ends when the last keypoint gather has finished
        e1.record(st)
        torch.cuda.synchronize()
        wall = time.time() - t0
        ms_dev = e0.elapsed_time(e1)
        if profile:
            engine.set_profiling(False)
        launches = engine.launch_count + parser.launch_count - l0
        barrier()
        ms = max(ms_dev, 0.0)
        # host-synchronous paths are bounded by wall clock, device-async ones by the stream events: take the larger
        ms = max(ms, wall * 1e3) if fn is not step_device else ms
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), launches

    # sanity: the device path and the host path agree with each other before anything is timed
    step_device(0)
    ref_h = drain_device()
    torch.cuda.synchronize()
    if ref_h is None:
        ref_h = parser.fetch(BATCH, cap=HCAP)
    step_host(0)
    host_h = drain_host()
    assert all(a.tobytes() == b.tobytes() for a, b in zip(ref_h, host_h)), "device and host paths disagree"
    n_humans = sum(len(h) for h in host_h)

    sampler = ClockSampler(local_rank)
    if rank == 0 and headline:
        sampler.start()
    # sustained pre-load: >= 2 s of the same steps before anything is timed, so that the power-cap state of the timed
    # region is the steady one (every rank: the steps contain the collective); nvidia-smi also needs ~0.3 s for its first sample
    t_pre = time.time()
    n_pre = 0
    pre_target = 2.0 if headline else 0.5
    while True:
        for i in range(10):
            step_device(n_pre + i)
        n_pre += 10
        drain_device()
        torch.cuda.synchronize()
        flag = torch.tensor([1.0 if time.time() - t_pre < pre_target else 0.0], device=dev)
        if world > 1:
            dist.all_reduce(flag, op=dist.ReduceOp.MAX)
        if flag.item() == 0.0 or n_pre >= 2000:
            break
    sampler.lines.clear()                   # keep only samples taken under load
    # pass A: the timed K steps, per-op profiling OFF -> value
    ms_total, launches = timed(step_device, steps, warmup)
    clocks = sampler.stop() if rank == 0 and headline else None
    if args.dump_outputs and rank == 0:
        dump_humans(args.dump_outputs, f"{key}_{args.dtype}", dpend.pop("last") if use_graph else parser.fetch(BATCH, cap=HCAP), HCAP)
    # pass B: the same K steps with per-op CUDA events on the launching stream -> kernel time for the roofline
    saved_graph = use_graph
    use_graph = False                       # per-op events need the kernels launched one by one
    for i in range(3):
        step_device(i)
    pstate["events"] = []
    ms_prof, _ = timed(step_device, steps, 0, profile=True)
    parse_events = pstate["events"]
    pstate["events"] = None
    use_graph = saved_graph
    prof_ms, prof_ty, prof_fl, prof_runs = engine.get_profile()
    parse_ms_events = float(np.mean([a.elapsed_time(b) for a, b in parse_events])) if parse_events else None
    e2e_steps = max(3, steps)
    ms_e2e, _ = timed(step_host, e2e_steps, max(3, warmup))
    # the synchronous form of the same public call (one batch in flight), for the record
    sync_steps = max(3, steps // 2)
    if PIFPAF:
        def step_sync(i):       # one batch in flight: submit + collect
            return engine.collect_pose(engine.submit_pose(parser, frames_np[i % N_INPUT_SETS]), cap=HCAP)
    else:
        def step_sync(i):
            return engine.run_pose(parser, frames_np[i % N_INPUT_SETS], cap=HCAP)
    ms_sync, _ = timed(step_sync, sync_steps, 3)
    ms_sync = max(ms_sync, 1e-6)

    frames_total = world * BATCH * steps
    value = frames_total / (ms_total / 1e3)
    e2e_value = world * BATCH * e2e_steps / (ms_e2e / 1e3)

    # parser alone on device-resident tensors at several batch sizes (launch-bound at small batches: SURVEY 8d)
    parse_sweep = None
    if headline and not PIFPAF and rank == 0:
        parse_sweep = []
        for nb in (16, 64, 128):
            reps = nb // BATCH if nb >= BATCH else 1
            cbig = d_conf.repeat(reps, 1, 1, 1)[:nb].contiguous(); pbig = d_paf.repeat(reps, 1, 1, 1)[:nb].contiguous()
            p2 = capi.PafParser(0.05, 0.05, device=local_rank)
            p2.set_capacity(peaks_per_part=128, candidates_per_limb=2048, humans=HCAP)
            for _ in range(3):
                p2.process_device(cbig.data_ptr(), pbig.data_ptr(), nb, 19, 38, HF, WF, st.cuda_stream)
            torch.cuda.synchronize()
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            reps_t = 20
            e0.record(st)
            for _ in range(reps_t):
                p2.process_device(cbig.data_ptr(), pbig.data_ptr(), nb, 19, 38, HF, WF, st.cuda_stream)
            e1.record(st)
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / reps_t
            parse_sweep.append({"frames": nb, "ms": ms, "frames_per_s": nb / (ms / 1e3)})
            p2.close()
            del cbig, pbig

    line = None
    if rank == 0:
        peaks, peak_src = load_peaks()
        conv_ms = float(prof_ms[prof_ty == models.OP_CONV].sum())
        other_ms = float(prof_ms[prof_ty != models.OP_CONV].sum())
        n_conv = int((prof_ty == models.OP_CONV).sum())
        algo_flops = ALGO_FLOPS_PER_FRAME * BATCH
        achieved = algo_flops / (conv_ms / 1e3) / 1e12 if conv_ms > 0 else 0.0
        if args.dtype == "tf32":
            peak = float(peaks.get("tf32_tflops_sustained", 0.5 * float(peaks.get("bf16_tflops_sustained", 1400.0))))
            peak_note = (f"{peak_src} tf32_tflops_sustained" if "tf32_tflops_sustained" in peaks else
                         f"half of the {peak_src} bf16_tflops_sustained (kind::tf32 issues K=8 per instruction against K=16 for f16/bf16: the tensor pipe's TF32 rate is half its 16-bit rate)")
        else:
            peak = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1400.0)))
            peak_note = f"{peak_src} bf16_tflops_sustained (kernel timed inside a long step)"
        traffic, traffic_source = None, None
        tpath = os.path.join(ROOT, "profiles", "conv_traffic.json")
        if os.path.exists(tpath) and key == "cfg3" and args.dtype == "f16":      # the ncu capture is of the headline workload only
            try:
                tj = json.load(open(tpath))
                traffic = tj.get("dram_bytes_per_step")
                traffic_source = tj.get("source", "ncu capture committed under profiles/ (not measured in this run)")
            except Exception:
                traffic = None
        h2d = BATCH * IN_H * IN_W * 3
        d2h = BATCH * HCAP * rec_bytes + BATCH * 8
        cfg = bench_config(world)
        line = {
            "metric": METRIC(), "value": value, "unit": "frames/s",
            "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": ms_total / steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": ("tf32 operands (fp32 activations in HBM), f32 accumulate (conv); f32/f64 (parse)" if args.dtype == "tf32"
                      else "f16 operands, f32 accumulate (conv); f32/f64 (parse)"), "data": "synthetic",
            "config": cfg,
            "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                    "api": ("hp_pose_submit_pifpaf_u8_host / hp_pose_collect (pinned host frames in, human_t records out, two batches in flight: the decoder runs on its own stream under the next batch's convs)" if PIFPAF else
                            "hp_pose_submit_u8_host / hp_pose_collect (pinned host frames in, human_t records out, two batches in flight, CUDA-graph replay)"),
                    "synchronous_call": {"value": world * BATCH * sync_steps / (ms_sync / 1e3), "api": "submit + collect, one batch in flight" if PIFPAF else "hp_pose_run_u8_host (one batch in flight)"},
                    "graphs": engine.pose_stats()},
            "gpu_launches": int(launches),
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak if peak else None,
                         "traffic": traffic, "traffic_source": traffic_source,
                         "kernel": "conv_tcgen05 family (conv_tcgen05_kernel / _swap_kernel / conv_halo_kernel / conv_stem3_kernel)", "launches_per_step": n_conv,
                         "algorithmic_flops_per_step": algo_flops, "kernel_ms_per_step": conv_ms,
                         "kernel_share_of_step": conv_ms / (ms_prof / steps), "peak_source": peak_note,
                         "timing": f"per-op CUDA events on the launching stream over a second pass of the same {steps} steps ({ms_prof / steps:.3f} ms/step with the events; `value` is timed without them)"},
            "clocks": clocks,
            "sustained_preload": {"steps": n_pre, "seconds": pre_target},
        }
        # SURVEY 8d: backbone-only and parser-only rates of the same run (per GPU), and the parser against its HBM bound
        step_ms = ms_prof / steps
        parse_ms = parse_ms_events if parse_ms_events else max(step_ms - conv_ms - other_ms, 1e-6)
        hbm = float(peaks.get("hbm_gbs", 6650.0))
        # SURVEY 8d: (19+38)*Hf*Wf*4 B per frame for conf/PAF; (17*5+19*9)*h*w*4 B for the PIF/PAF fields
        frame_bytes = ((17 * 5 + 19 * 9) if PIFPAF else 57) * HF * WF * 4
        parse_bytes = BATCH * frame_bytes
        line["breakdown"] = {"backbone_ms_per_step": conv_ms + other_ms, "backbone_frames_per_s": BATCH / ((conv_ms + other_ms) / 1e3),
                             "parse_ms_per_step": parse_ms, "parse_frames_per_s": BATCH / (parse_ms / 1e3),
                             "parse_hbm_frac": (parse_bytes / (parse_ms / 1e3) / 1e9 / hbm) if parse_bytes else None,
                             "parse_algorithmic_bytes_per_step": parse_bytes,
                             "note": "parse = CUDA events around the parser's launches (counter memset + 2 kernels) inside the step, mean over the steps of the second pass; its HBM bound counts only the network-output tensors read once"}
        if parse_sweep:
            for e in parse_sweep:
                e["hbm_frac"] = e["frames"] * frame_bytes / (e["ms"] / 1e3) / 1e9 / hbm
            line["breakdown"]["parse_alone_by_batch"] = parse_sweep
        layers = [{"op": i, "name": graph.ops[i].name, "type": int(prof_ty[i]), "ms": float(prof_ms[i]),
                   "tflops": (float(prof_fl[i]) * BATCH / (prof_ms[i] / 1e3) / 1e12 if prof_ms[i] > 0 and prof_fl[i] > 0 else None)}
                  for i in range(len(prof_ms))]
        if args.layers_dir:
            os.makedirs(args.layers_dir, exist_ok=True)
            with open(os.path.join(args.layers_dir, f"bench_layers_{key}_{args.dtype}_n{world}.json"), "w") as f:
                json.dump({"ms_per_step": ms_total / steps, "conv_ms": conv_ms, "other_engine_ms": other_ms, "profiled_runs": prof_runs, "layers": layers}, f, indent=1)
        # bounded CPU baseline (rank 0, N=1, headline only): the reference parser on the host cores + the conv port
        if world == 1 and headline and not args.no_cpu_baseline and not PIFPAF:
            cores = cpu_threads()
            threads = min(cores, BATCH)
            rate, kind = cpu_parse_rate(conf_np, paf_np, 10.0, threads)
            conv_one, conv_threads = cpu_conv_port(WL["graph"], 1)
            conv_one()                                   # warm-up (allocations, oneDNN primitive caches)
            tc0 = time.time(); n_cpu_frames = 0
            while n_cpu_frames < 2 or (time.time() - tc0 < 6.0 and n_cpu_frames < 16):
                conv_one(); n_cpu_frames += 1
            conv_s = (time.time() - tc0) / n_cpu_frames
            whole = 1.0 / (conv_s + 1.0 / rate)
            line["cpu_baseline"] = {"value": whole, "unit": "frames/s", "cores": max(threads, conv_threads), "kind": "port",
                   "sample": f"conv stage: {n_cpu_frames} frames {IN_H}x{IN_W} through a PyTorch fp32 port of the same graph, torch.set_num_threads({conv_threads}) ({conv_s * 1e3:.0f} ms/frame; the reference's "
                             f"convs are TensorRT-on-GPU, no CPU implementation exists) + parse stage: 10 s of the reference CPU parser (src/paf.cpp via oracle/_ref) on the step's {BATCH} synthetic "
                             f"{HF}x{WF} crowd frames, {threads} threads of {cores} usable host threads",
                   "parse_only": {"value": rate, "unit": "frames/s", "cores": threads, "kind": kind}}
            gpu_parse = max(parse_sweep, key=lambda e: e["frames_per_s"]) if parse_sweep else None
            line["parse_only"] = {"gpu": {"value": BATCH / (parse_ms / 1e3), "unit": "frames/s", "what": f"parse stage inside the step, batch {BATCH}"},
                                  "gpu_best_batch": gpu_parse,
                                  "cpu_reference": {"value": rate, "unit": "frames/s", "cores": threads, "kind": kind, "what": "the reference's own src/paf.cpp, one replica per thread"},
                                  "ratio_in_step": BATCH / (parse_ms / 1e3) / rate}
        line["humans_per_batch"] = n_humans
    engine.close()
    parser.close()
    del frames_dev, frames_host, d_conf, d_paf
    import gc
    gc.collect()
    torch.cuda.empty_cache()
    return line


def run_ours(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    ctx = (rank, local_rank, world, dev)
    line = measure(args, args.workload, ctx, headline=True)
    # the other single-GPU BASELINE configs in the same run (N=1 only): one entry each under `extra_configs`
    if world == 1 and args.workload == "cfg3" and args.dtype == "f16" and not args.no_extra:
        extra = []
        for key in ("cfg2", "cfg4", "cfg5"):
            try:
                e = measure(args, key, ctx, headline=False)
                extra.append({k: e[k] for k in ("metric", "value", "unit", "ms_per_step", "steps", "config", "e2e", "roofline", "breakdown", "gpu_launches")})
            except Exception as ex:      # an extra config must never cost the headline line
                extra.append({"workload": key, "error": repr(ex)})
        line["extra_configs"] = extra
        if not args.no_tf32_line:
            try:
                a2 = argparse.Namespace(**vars(args)); a2.dtype = "tf32"
                e = measure(a2, "cfg3", ctx, headline=False)
                line["tf32"] = {k: e[k] for k in ("metric", "value", "unit", "ms_per_step", "steps", "dtype", "e2e", "roofline", "gpu_launches")}
            except Exception as ex:
                line["tf32"] = {"error": repr(ex)}
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dtype", default="f16", choices=["f16", "tf32"], help="conv arithmetic: f16 = data_type::kHALF, tf32 = data_type::kFLOAT of the reference API (tensorrt.hpp:14-22)")
    ap.add_argument("--no-graph", action="store_true", help="device-resident steps launch every kernel on the stream instead of replaying the captured CUDA graph")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra_configs entries (cfg2 / cfg4 / cfg5) of the default run")
    ap.add_argument("--no-tf32-line", action="store_true", help="skip the tf32 entry of the default run")
    ap.add_argument("--workload", default="cfg3", choices=sorted(WORKLOADS), help="BASELINE.json config (default: the headline cfg3)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the keypoint records of the last timed step of every measured config to "
                    "DIR/<config>_<dtype>_human_*.npy; they come from the synthetic parser inputs, not from the convs (see dump_humans)")
    ap.add_argument("--layers-dir", metavar="DIR", help="write the per-op CUDA-event times of every measured config to DIR/bench_layers_*.json")
    args = ap.parse_args()
    select_workload(args.workload)
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
