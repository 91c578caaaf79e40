#!/usr/bin/env python3
"""bench.py -- decode Mpixels/s of the VarDCT transform pipeline on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload NAME] [--dump-outputs DIR]

One "step" = one pass of the hot path (dequant+CfL+LLF+IDCT -> Gaborish -> EPF -> XYB->linear RGB)
over one frame of synthetic content.

  value     whole-job Mpixels/s with the coefficient groups + side info already resident in HBM
            (CUDA events on the launch stream, K steps, max over ranks).
  e2e       the same metric through the C ABI with HOST buffers: every step does frame_begin
            (side-info H2D) + submit_group per AC group (pinned H2D) + frame_finish (kernels + D2H of
            the pixels into pinned host memory).
  roofline  dominant kernel: algorithmic bytes per launch / its CUDA-event time, vs measured HBM peak.
  cpu_baseline  the reference's own CPU code for the same hot path (DecodeGroupForRoundtrip + its
            render-pipeline stages, oracle/_ref built from /root/reference) on all host cores.

N > 1 (launched by torchrun, one rank per GPU): the frame is sharded into bands of AC-group rows;
every rank inverse-transforms and filters its band (plus the varblocks touching its 7-row halo) and the
bands are all-gathered over NCCL so that every GPU holds the full frame ("scaling": "strong").
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

WORKLOADS = {
    # name: (w, h, distance, effort, gaborish, epf, kind)  -- -1 = encoder default for the distance
    "8k-d1": (7680, 4320, 1.0, 7, -1, -1, "photo"),          # metric: 8K VarDCT d1.0 (gab on, epf 1)
    "8k-d0.5-full": (7680, 4320, 0.5, 7, 1, 3, "photo"),     # BASELINE config 3
    "4k-d1": (4096, 4096, 1.0, 7, -1, -1, "photo"),          # BASELINE config 2
    "1080p-d1": (1920, 1080, 1.0, 7, -1, -1, "photo"),
    "512-d1": (512, 512, 1.0, 7, -1, -1, "photo"),
    # BASELINE config 4: 16384^2 uniform-noise image, d2.0, EPF iters 3 (gab on at d2) -- sharded over 8 GPUs
    "16k-d2-epf3": (16384, 16384, 2.0, 7, -1, 3, "noise"),
    # BASELINE config 2, second half: synthetic frame whose AcStrategy map cycles through all 27 transforms
    # (cjxl never emits > 64x64, SURVEY.md §8c caveat); coefficients int16 Laplace, gab + 3 EPF passes
    "4k-all27": (4096, 4096, None, None, 1, 3, "synthetic-all-strategies"),
    # BASELINE config 5: 64 independent 1920x1080 frames, frame-per-GPU replicas (no collective): --workload 64x1080p
    "64x1080p": (1920, 1080, 1.0, 7, -1, -1, "photo"),
}
BIG = {"16k-d2-epf3"}   # no cached copy of the reference decoder's pixels (3.2 GB): parity vs the reference hot path


OUTPUT_TEXT = {"f32": "interleaved linear RGB f32 (12 B/px)",
               "srgb8": "interleaved sRGB 8-bit, FromLinear + dithered WriteToOutput as djxl writes it (3 B/px)"}


def log(*a):
    print("[bench]", *a, file=sys.stderr, flush=True)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the timed region runs (B200_PROFILING.md)."""

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        # samples under load = upper half of the SM clock samples
        sm_sorted = sorted(sm)
        load = sm_sorted[len(sm_sorted) // 2:] if sm_sorted else []
        return {"sm_mhz": float(np.median(load)) if load else None,
                "sm_max_mhz": max(mx) if mx else None, "samples": len(sm), "reasons": sorted(reasons)}


def prepare_frame(name: str, rank: int, world: int, barrier):
    """Workload preparation (untimed): the reference (oracle/_ref) plays the host libjxl --
    synthetic image -> bitstream -> entropy-decoded coefficient groups + side info. Rank 0
    builds the cache file, the other ranks load it."""
    import jxl_workload as wl
    from oracle import ref
    w, h, dist, effort, gab, epf, kind = WORKLOADS[name]
    source = "reference-encoded"
    if kind == "synthetic-all-strategies":
        desc, coeffs = wl.synthetic_frame(w, h, seed=1234, gab=gab, epf_iters=epf)
        return dict(desc=desc, coeffs=coeffs, jxl=None, hist=wl.strategy_histogram(desc.ac_strategy), bpp=None,
                    decoded=None), "synthetic coefficients, every AcStrategy"
    if not ref.available():
        log("oracle/_ref missing: falling back to a synthetic all-strategy frame")
        desc, coeffs = wl.synthetic_frame(w, h, seed=1234)
        return dict(desc=desc, coeffs=coeffs, jxl=None, hist=wl.strategy_histogram(desc.ac_strategy), bpp=None,
                    decoded=None), "synthetic-coefficients"
    if rank == 0:
        t = time.time()
        fr = wl.reference_frame(w, h, dist, effort, gab, epf, seed=1234, kind=kind, cache=True,
                                want_decoded=name not in BIG, threads=host_cpu_info()["cores"])
        log(f"frame ready in {time.time() - t:.1f}s: {w}x{h} d{dist} e{effort} gab={fr['desc'].gab} "
            f"epf={fr['desc'].epf_iters} bpp={fr['bpp']:.2f} ac_type={'int16' if fr['desc'].ac_type == 0 else 'int32'}")
    barrier()
    if rank != 0:
        fr = wl.reference_frame(w, h, dist, effort, gab, epf, seed=1234, kind=kind, cache=True,
                                want_decoded=name not in BIG)
    return fr, source


def bind_near_gpu(index: int) -> str:
    """Pin this process (and so its page-locked buffers, first touch) to the CPUs of the GPU's NUMA node -- what
    `numactl` does for a production decoder.  A host buffer on the far socket halves the PCIe rates of the e2e
    arm (seen as 2x run-to-run differences on the same box before this was here).  Returns a note for the log."""
    try:
        import pynvml
        import torch
        pynvml.nvmlInit()
        pr = torch.cuda.get_device_properties(index)
        try:   # the physical device behind this CUDA index (CUDA_VISIBLE_DEVICES may renumber)
            h = pynvml.nvmlDeviceGetHandleByPciBusId(
                f"{pr.pci_domain_id:08x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0".encode())
        except Exception:  # noqa: BLE001
            h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        near = {i for i in range(os.cpu_count()) if (words[i // 64] >> (i % 64)) & 1}
        allowed = os.sched_getaffinity(0)
        cpus = near & allowed
        if cpus and cpus != allowed:
            os.sched_setaffinity(0, cpus)
            return f"bound to {len(cpus)} CPUs near GPU {index}"
        return f"no binding needed ({len(allowed)} CPUs allowed, {len(near)} near GPU {index})"
    except Exception as e:  # noqa: BLE001
        return f"no NUMA binding ({e!r})"


def host_cpu_info() -> dict:
    """Cores this process may actually use: the scheduler affinity mask capped by the cgroup CPU quota
    (os.cpu_count() reports the whole host, which a 1-GPU lease does not own)."""
    import math
    total = os.cpu_count() or 1
    try:
        aff = len(os.sched_getaffinity(0))
    except AttributeError:
        aff = total
    quota = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    quota = float(txt[0]) / float(txt[1])
            else:
                q = float(txt[0])
                if q > 0:
                    quota = q / float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            break
        except Exception:  # noqa: BLE001
            continue
    eff = aff if quota is None else max(1, min(aff, int(math.ceil(quota))))
    return {"cores": eff, "affinity": aff, "cgroup_quota": quota, "os_cpu_count": total}


DUMP_BYTES = 60_000_000   # --dump-outputs: what one run writes stays under 64 MB with the .npy headers


def output_sample(kind: str, frame: np.ndarray, budget: int) -> dict[str, np.ndarray]:
    """What --dump-outputs writes for one output kind: the whole frame as float32 when it fits in `budget`
    bytes, otherwise a fixed sample (seed 0, so two runs of the same workload pick the same samples) with its
    flat indices as float64 (exact below 2**53)."""
    if frame.size * 4 <= budget:
        return {kind: frame.astype(np.float32)}
    idx = np.unique(np.random.default_rng(0).integers(0, frame.size, budget // 12))
    return {kind: frame.reshape(-1)[idx].astype(np.float32), f"{kind}_index": idx.astype(np.float64)}


def geomean_excluding_first(secs, px: int) -> float:
    """Mpixel/s as tools/speed_stats.cc:37-57 reports it: geometric mean over the repetitions, the
    first one excluded (when there is more than one)."""
    v = [px / float(t) / 1e6 for t in secs]
    if len(v) > 1:
        v = v[1:]
    return float(np.exp(np.mean(np.log(v))))


def workload_text(name: str, desc, source: str, output: str) -> str:
    """The one description of the workload both arms print (same frame, same hot path, same output)."""
    w, h, dist, effort, _, _, _ = WORKLOADS[name]
    es = "int16" if desc.ac_type == 0 else "int32"
    enc = f"VarDCT d{dist} e{effort}" if dist is not None else "VarDCT"
    return (f"{name}: {w}x{h} {enc}, gab={desc.gab} epf_iters={desc.epf_iters}, {source}, "
            f"coefficients {es} as the reference decoder chose, hot path = dequant+IDCT -> Gaborish/EPF -> XYB->RGB, "
            f"output {OUTPUT_TEXT[output]}")


def cpu_reference_numbers(fr, w: int, h: int, output: str, reps: int, threads_list) -> dict:
    """The reference's own hot-path code (oracle/_ref) on `threads` host threads for each entry of
    threads_list: {threads: {"f32": Mpx/s, "srgb8": Mpx/s}} + the whole decoder (entropy decode incl.)."""
    from oracle import ref
    out = {"hot": {}, "full": {}}
    for nt in threads_list:
        frame = ref.Frame(fr["jxl"], nt)
        r = max(2, reps if nt > 1 else min(reps, 3))
        by = {}
        for kind in ("f32", "srgb8"):
            if kind != output and nt == 1:
                continue
            if kind == "f32":
                _, secs = frame.render(-1, reps=r + 1, want_output=False)
            else:
                _, secs = frame.render_out(-33, 2, reps=r + 1, want_output=False)
            by[kind] = geomean_excluding_first(secs, w * h)
        frame.close()
        out["hot"][nt] = by
        runner = ref.Runner(nt)
        buf = np.empty((h, w, 3), np.float32)
        ts = []
        for _ in range(3 if nt > 1 else 2):
            t0 = time.perf_counter()
            ref.decode_linear_f32(fr["jxl"], nt, buf, runner)
            ts.append(time.perf_counter() - t0)
        runner.close()
        out["full"][nt] = geomean_excluding_first(ts, w * h)
    return out


def algorithmic_bytes(desc, rows: int, out_px_bytes: int = 12) -> dict:
    """DESIGN.md §Roofline: bytes one launch must move, per kernel, for `rows` pixel rows."""
    px = desc.xsize * rows
    es = 2 if desc.ac_type == 0 else 4
    side = 21.0 / 64.0  # acs 1 + quant 4 + sigma 4 + dc 12 bytes per 8x8 block
    return {"idct": px * (3 * es + side + 12), "filter": px * (12 + out_px_bytes + 4.0 / 64),
            "fused_path": px * (3 * es + side + out_px_bytes)}


def run_reference(args, rank: int) -> int:
    """--impl reference: the reference's own CPU implementation of the hot path (not the whole
    decoder: entropy decoding is outside the path) on every host core this process may use, same frame.
    `steps` timed passes (+1 untimed first one, speed_stats.cc semantics)."""
    if rank != 0:
        return 0
    import jxl_workload as wl
    from oracle import ref
    name = args.workload
    w, h, dist, effort, gab, epf, kind = WORKLOADS[name]
    cpu = host_cpu_info()
    cores = cpu["cores"]
    fr = wl.reference_frame(w, h, dist, effort, gab, epf, seed=1234, kind=kind, cache=True)
    frame = ref.Frame(fr["jxl"], cores)

    def hot(kind, reps):
        if kind == "f32":   # ... XYB -> linear RGB, planar float image (the path's §8 scope)
            return frame.render(-1, reps=reps, want_output=False)[1]
        # ... + FromLinear (sRGB) + WriteToOutput into an interleaved 8-bit buffer (what djxl writes)
        return frame.render_out(-33, 2, reps=reps, want_output=False)[1]

    hot(args.output, max(1, args.warmup))
    secs = hot(args.output, args.steps + 1)
    other = "srgb8" if args.output == "f32" else "f32"
    other_secs = hot(other, max(3, min(args.steps, 8)) + 1)
    frame.close()
    mps = geomean_excluding_first(secs, w * h)
    other_mps = geomean_excluding_first(other_secs, w * h)
    one = cpu_reference_numbers(fr, w, h, args.output, 3, [1])
    many_full = cpu_reference_numbers(fr, w, h, args.output, 2, [cores])["full"][cores] if cores > 1 else one["full"][1]
    line = {
        "impl": "reference", "metric": "decode_mpixels_per_s", "value": mps, "unit": "Mpixel/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * w * h / (mps * 1e6), "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_text(name, fr["desc"], "reference-encoded", args.output)},
        "variants": {other: {"value": other_mps, "unit": "Mpixel/s", "output": OUTPUT_TEXT[other]}},
        "cpu_baseline": {"value": mps, "unit": "Mpixel/s", "cores": cores, "kind": "reference",
                         "host": cpu, "hwy_target": ref.hwy_target(),
                         "sample": f"{args.steps} passes (+1 untimed first) of DecodeGroupForRoundtrip + the reference's "
                                   f"Gaborish/EPF/XYB stages over the full {w}x{h} frame; geomean excluding the first "
                                   "(tools/speed_stats.cc:37-57)",
                         "one_thread_mpixels_per_s": one["hot"][1][args.output],
                         "full_decode_mpixels_per_s": many_full,
                         "full_decode_one_thread_mpixels_per_s": one["full"][1]},
        "e2e": {"value": mps, "unit": "Mpixel/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


def run_replicas(args, rank: int, local_rank: int, world: int) -> int:
    """BASELINE config 5: a batch of 64 independent 1920x1080 frames, frame-per-GPU (round-robin over the
    ranks, no collective -- SURVEY.md §8e "replicas only").  value = whole-batch Mpixel/s with the coefficients
    resident in HBM (every frame still does its own frame_begin: side-info upload + plan); e2e = host
    coefficient blocks -> host pixels through the C ABI; latency = per-frame wall time of the e2e call
    sequence (frame_begin .. frame_finish) on an otherwise idle GPU, p50 over the rank's frames."""
    import torch
    import torch.distributed as dist

    import jxl_workload as wl
    from libjxl_b200 import abi, pipeline
    from oracle import ref
    torch.cuda.set_device(local_rank)
    log(f"rank {rank}: {bind_near_gpu(local_rank)}")
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()

    w, h, dist_, effort, gab, epf, kind = WORKLOADS["64x1080p"]
    NF = 64
    mine = list(range(rank, NF, world))
    t0 = time.time()
    if rank == 0:   # build the cache files once
        for i in range(NF):
            wl.reference_frame(w, h, dist_, effort, gab, epf, seed=i, kind=kind, cache=True, threads=host_cpu_info()["cores"])
    barrier()
    frames = [wl.reference_frame(w, h, dist_, effort, gab, epf, seed=i, kind=kind, cache=True) for i in mine]
    log(f"rank {rank}: {len(frames)} frames ready in {time.time() - t0:.1f}s")
    pipe = pipeline.TransformPipeline(device=local_rank, num_host_threads=1)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    # a 1080p frame fills about a quarter of the SMs: NPIPE contexts on their own streams keep several
    # frames in flight (device-resident throughput number); the e2e / latency loop below uses one context
    NPIPE = 4
    pipes = [pipe] + [pipeline.TransformPipeline(device=local_rank, num_host_threads=1) for _ in range(NPIPE - 1)]
    side = [torch.cuda.Stream() for _ in range(NPIPE)]
    ev_start = torch.cuda.Event()
    ev_side = [torch.cuda.Event() for _ in range(NPIPE)]
    descs = [pipeline.pin_side_info(f["desc"]) for f in frames]
    dev = [torch.from_numpy(f["coeffs"]).cuda() for f in frames]
    ptrs = [[d[c].data_ptr() for c in range(3)] for d in dev]
    outs = [torch.empty((h, w, 3), dtype=torch.float32, device="cuda") for _ in frames]
    row_bytes = w * 12

    def batch_device():
        ev_start.record(stream)
        for q in range(NPIPE):
            side[q].wait_event(ev_start)
        for i, d in enumerate(descs):
            q = i % NPIPE
            pipes[q].set_device_coefficients(ptrs[i])
            pipes[q].frame_begin(d)
            pipes[q].render_device(outs[i].data_ptr(), row_bytes, side[q].cuda_stream)
        for q in range(NPIPE):   # join: the timing events live on `stream`
            ev_side[q].record(side[q])
            stream.wait_event(ev_side[q])

    for _ in range(max(3, args.warmup)):
        batch_device()
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    barrier()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = sum(p_.launch_count() for p_ in pipes)
    ev0.record(stream)
    for _ in range(args.steps):
        batch_device()
    ev1.record(stream)
    torch.cuda.synchronize()
    barrier()
    launches = sum(p_.launch_count() for p_ in pipes) - launches0
    t = torch.tensor([ev0.elapsed_time(ev1)], device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / args.steps
    value = NF * w * h / (ms_step * 1e-3) / 1e6
    # parity of every frame of this rank against the reference decoder's pixels
    peak = 0.0
    for i, f in enumerate(frames):
        peak = max(peak, float(np.abs(outs[i].cpu().numpy() - f["decoded"]).max()))

    # ---- end to end: host coefficient blocks -> host pixels, frame by frame ----
    for p_ in pipes[1:]:
        p_.close()
    pipe.set_device_coefficients(None)
    host = []
    h2d = d2h = 0
    for f, d in zip(frames, descs):
        blk = pipeline.pinned_array((d.num_groups, 3, abi.GROUP_COEFFS), f["coeffs"].dtype)
        groups = {}
        for g in range(d.num_groups):
            n = d.group_ncoeff(g)
            blk[g] = f["coeffs"][:, g]
            groups[g] = [blk[g, c, :n] for c in range(3)]
            h2d += (2 * abi.GROUP_COEFFS + n) * f["coeffs"].dtype.itemsize
        yb, xb = d.ysize_blocks, d.xsize_blocks
        h2d += yb * xb * (1 + 4 + 1 + 12) + d.dequant.nbytes + 2 * d.ytox.size
        out = pipeline.pinned_array((h, w, 3), np.float32)
        d2h += out.nbytes
        host.append((pipe.make_batch(list(range(d.num_groups)), groups), out, blk))

    def one_frame(i):
        pipe.frame_begin(descs[i])
        pipe.frame_set_output(host[i][1])
        pipe.submit_batch(host[i][0], 0)
        pipe.frame_finish(host[i][1])

    for i in range(len(frames)):
        one_frame(i)
    barrier()
    lat = []
    n_e2e = max(2, min(args.steps, 5))
    t0 = time.perf_counter()
    for _ in range(n_e2e):
        for i in range(len(frames)):
            a = time.perf_counter()
            one_frame(i)
            lat.append(time.perf_counter() - a)
    barrier()
    e2e_s = (time.perf_counter() - t0) / n_e2e
    te = torch.tensor([e2e_s], device="cuda")
    lat_t = torch.tensor([float(np.median(lat)), float(np.percentile(lat, 95))], device="cuda")
    by = torch.tensor([float(h2d), float(d2h), peak], device="cuda")
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
        dist.all_reduce(lat_t, op=dist.ReduceOp.MAX)
        by2 = by.clone()
        dist.all_reduce(by2)
        dist.all_reduce(by, op=dist.ReduceOp.MAX)
        by[0], by[1] = by2[0], by2[1]
    clocks = sampler.stop() if rank == 0 else None
    pipe.close()
    if rank == 0:
        line = {
            "metric": "decode_mpixels_per_s", "value": value, "unit": "Mpixel/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"64x1080p: batch of {NF} independent {w}x{h} VarDCT d{dist_} e{effort} frames (seeds 0..{NF - 1}), "
                                   "frame-per-GPU replicas round-robin over the ranks, no collective; one step = the whole batch; "
                                   "output interleaved linear RGB f32",
                       "parallelism": f"{world} x replicas", "frames_per_rank": len(mine), "contexts_per_rank": NPIPE,
                       "l2": f"batch working set per rank {len(mine) * (3 * frames[0]['coeffs'][0].nbytes + 2 * w * h * 12) / 1e6:.0f} MB"},
            "e2e": {"value": NF * w * h / float(te.item()) / 1e6, "unit": "Mpixel/s", "h2d_bytes_per_step": int(by[0].item()),
                    "d2h_bytes_per_step": int(by[1].item()), "steps": n_e2e, "submit": "dense",
                    "how": "per frame: frame_begin + frame_set_output + submit_groups (all groups, pinned host blocks) + frame_finish"},
            "latency_ms": {"p50": 1e3 * float(lat_t[0].item()), "p95": 1e3 * float(lat_t[1].item()),
                           "what": "host coefficients -> host pixels of one 1080p frame (max over ranks of the per-rank percentiles)"},
            "gpu_launches": int(launches), "clocks": clocks,
            "parity": {"peak_abs_err_vs_reference": float(by[2].item()), "frames_checked": NF},
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="8k-d1", choices=list(WORKLOADS))
    ap.add_argument("--output", default="f32", choices=["f32", "srgb8"],
                    help="pixel format the path ends in: linear f32 (the §8 scope, default) or sRGB 8-bit "
                         "(sRGB transfer function + WriteToOutput packing fused into the filter kernel's store); "
                         "the other one is measured too and reported under \"variants\"")
    ap.add_argument("--submit", default="sparse", choices=["dense", "sparse"],
                    help="e2e arm: sparse = the non-zero lists of jxlgpu_submit_groups_sparse, which the compiled "
                         "libjxl integration (integration/patch_libjxl.py: the patched DecodeACVarBlock appends them "
                         "while it entropy-decodes; tests/test_integration_libjxl.py) hands over -- default; dense = "
                         "[group][3][65536] coefficient blocks in libjxl's ACImage layout.  The other one is measured "
                         "too and reported under \"variants\"")
    ap.add_argument("--no-variants", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--gather", default="auto", choices=["auto", "ce", "sm", "multicast", "p2p", "nccl"],
                    help="N>1: how the bands are all-gathered into every rank's frame buffer (symmetric memory): ce = finished "
                         "row chunks travel to the peers through the copy engines while the next chunk is filtered; sm = the same "
                         "chunks stored to all peers by a copy kernel; p2p: peer stores fused into the filter kernel; multicast: "
                         "multimem.st through the NVSwitch; nccl: all_gather_into_tensor after the kernels; auto (default) = ce, "
                         "except sm for the f32 frame on 4 and more GPUs (DESIGN.md section 6)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the frame of the last device-resident step of every measured "
                         "output kind to DIR/<kind>.npy as float32 (a seeded sample of at most 64 MB in all, with its "
                         "flat indices in DIR/<kind>_index.npy, when the whole frame does not fit)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or args.workload == "64x1080p"):
        ap.error("--dump-outputs is supported for the single-frame b200 path")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.gather in ("p2p", "multicast"):
        os.environ["JXLGPU_GATHER"] = "kernel"   # (read when the context is created)
    if args.gather == "sm":
        os.environ["JXLGPU_GATHER"] = "sm"       # peer_copy_kernel per row chunk instead of copy-engine copies

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        return run_reference(args, rank)
    if args.workload == "64x1080p":
        return run_replicas(args, rank, local_rank, world)

    import torch
    import torch.distributed as dist

    import jxl_workload as wl  # noqa: F401
    from libjxl_b200 import abi, pipeline, sharding

    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: the product path has no CPU fallback"}))
        return 2
    torch.cuda.set_device(local_rank)
    log(f"rank {rank}: {bind_near_gpu(local_rank)}")
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()

    fr, source = prepare_frame(args.workload, rank, world, barrier)
    desc, coeffs = fr["desc"], fr["coeffs"]
    W, H = desc.xsize, desc.ysize
    es = 2 if desc.ac_type == abi.AC_INT16 else 4
    if world > desc.ysize_groups:
        print(json.dumps({"error": f"{world} ranks but only {desc.ysize_groups} rows of AC groups to shard"}))
        return 2
    bands = sharding.band_partition(desc.ysize_groups, world)
    y0g, nyg = bands[rank]
    if world > 1:
        desc.band_y0_groups, desc.band_ny_groups = y0g, nyg
    band_y0, band_rows = sharding.band_pixel_rows(desc, y0g, nyg) if world > 1 else (0, H)
    need = sharding.groups_needed(desc, y0g, nyg) if world > 1 else list(range(desc.num_groups))
    max_rows = max(sharding.band_pixel_rows(desc, a, b)[1] for a, b in bands) if world > 1 else H

    n_submit_threads = 8
    pipe = pipeline.TransformPipeline(device=local_rank, num_host_threads=n_submit_threads)
    # a real (non-default) stream: the library launches on exactly this stream, so the
    # torch.cuda.Event pair below brackets its kernels (and NCCL's, which torch enqueues on it)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)

    def measure(kind: str, full: bool) -> dict:
        """Device-resident arm + (full: per-kernel pass, parity) + end-to-end arm for one output kind."""
        out_fmt = abi.OUT_RGB_F32 if kind == "f32" else abi.OUT_RGB_U8
        desc.out_format = out_fmt
        desc.stage_mask = 0 if kind == "f32" else abi.STAGE_SRGB
        tdtype = torch.float32 if kind == "f32" else torch.uint8
        ndtype = np.float32 if kind == "f32" else np.uint8
        isz = 4 if kind == "f32" else 1          # bytes per sample
        row_bytes = W * 3 * isz
        # ---------------- device-resident arm ----------------
        if "ptrs" not in shared:
            if world == 1:
                dev = torch.zeros((3, desc.num_groups, abi.GROUP_COEFFS), dtype=torch.int16 if es == 2 else torch.int32,
                                  device="cuda")
                dev.copy_(torch.from_numpy(coeffs))
                shared["ptrs"] = [dev[c].data_ptr() for c in range(3)]
            else:
                # only the groups this rank needs live on its GPU; the planes keep frame-wide indexing
                g0, g1 = min(need), max(need) + 1
                dev = torch.from_numpy(np.ascontiguousarray(coeffs[:, g0:g1])).cuda()
                shared["ptrs"] = [dev[c].data_ptr() - g0 * abi.GROUP_COEFFS * es for c in range(3)]
            shared["dev"] = dev
        pipe.set_device_coefficients(shared["ptrs"])
        pipe.frame_begin(desc)
        gather_mode = "none"
        hdl = None
        if world == 1:
            gathered = torch.empty((H, W, 3), dtype=tdtype, device="cuda")
            my_out = gathered
        else:
            slot = max_rows * W * 3
            gathered = None
            # auto: copy engines, except the f32 frame on 8 GPUs where NCCL measured 9 % faster (1.09 vs 1.19 ms:
            # nothing left to overlap the gather with; DESIGN.md §6)
            use_nccl = args.gather == "nccl"
            if args.gather == "auto":
                # measured (DESIGN.md §6): copy engines win while there is filter work to overlap with (N=2: 0.62 ms
                # vs sm 0.73, nccl 0.89); from 4 GPUs on the f32 frame is mostly gather: N=4 sm 0.85 / nccl 0.90 /
                # ce 0.99 ms, N=8 sm 1.04 / nccl 1.11 / ce 1.17
                if world >= int(os.environ.get("BENCH_AUTO_SM_MIN_WORLD", "4")) and kind == "f32":
                    os.environ["JXLGPU_GATHER"] = "sm"     # (read again by jxlgpu_set_output_replicas)
                else:
                    os.environ.pop("JXLGPU_GATHER", None)
            if not use_nccl:
                try:
                    # Fused compute + all-gather: the frame buffer of every rank is symmetric memory; a filter
                    # CTA writes its strip segment into the local slot and replays it to every peer with wide
                    # stores (multimem.st.v2 through the NVSwitch multicast mapping, or NVLink peer stores).
                    import torch.distributed._symmetric_memory as symm
                    flat = symm.empty(world * slot, dtype=tdtype, device=torch.device("cuda", local_rank))
                    hdl = symm.rendezvous(flat, dist.group.WORLD)
                    gathered = flat.view(world, max_rows, W, 3)
                    # measured on this box (N=2): peer stores 0.84 ms/step, multimem.st.v2 1.16 ms -> auto = p2p
                    mc = int(hdl.multicast_ptr) if args.gather == "multicast" else 0
                    if args.gather == "multicast" and not mc:
                        raise RuntimeError("multicast not supported here")
                    if mc:
                        pipe.set_output_replicas([], mc + rank * slot * isz)
                        gather_mode = "fused in the filter kernel: each CTA replays its finished region with multimem.st.v2 (NVSwitch multicast)"
                    else:
                        pipe.set_output_replicas([int(hdl.buffer_ptrs[p]) + rank * slot * isz for p in range(world) if p != rank])
                        gather_mode = ("fused in the filter kernel: each CTA replays its finished region to the peers (NVLink P2P float2 stores)"
                                       if args.gather == "p2p" else
                                       "SM copy kernel: every finished row chunk is stored to all peers' symmetric-memory frame buffers "
                                       "by peer_copy_kernel (16-byte NVLink stores) on a side stream while the next chunk is filtered"
                                       if args.gather == "sm" or os.environ.get("JXLGPU_GATHER") == "sm" else
                                       "copy engines: every finished row chunk is copied to the peers' symmetric-memory frame buffers "
                                       "(NVLink, cudaMemcpyAsync on side streams) while the next chunk is filtered")
                except Exception as e:  # noqa: BLE001
                    log(f"symmetric memory unavailable ({e!r}): falling back to NCCL all-gather")
                    hdl = None
                    gathered = None
            if gathered is None:
                gathered = torch.empty((world, max_rows, W, 3), dtype=tdtype, device="cuda")
                gather_mode = "NCCL all_gather_into_tensor after the filter kernel"
            my_out = gathered[rank]

        def whole_frame() -> np.ndarray:
            """The frame as rank 0 holds it: every band, as it arrived in its frame buffer."""
            if world == 1:
                return gathered.cpu().numpy()
            return np.concatenate([gathered[r, :sharding.band_pixel_rows(desc, *bands[r])[1]].cpu().numpy()
                                   for r in range(world)])

        def step():
            pipe.render_device(my_out.data_ptr(), row_bytes, stream.cuda_stream)
            if world > 1:
                if hdl is not None:
                    hdl.barrier(channel=0)      # publishes the peers' stores: the frame is complete everywhere
                else:
                    dist.all_gather_into_tensor(gathered.view(-1), my_out.reshape(-1))

        for _ in range(args.warmup):
            step()
        torch.cuda.synchronize()
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
        barrier()
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        launches0 = pipe.launch_count()
        ev0.record(stream)
        for _ in range(args.steps):
            step()
        ev1.record(stream)
        torch.cuda.synchronize()
        barrier()
        if args.dump_outputs and rank == 0:
            dumps.update(output_sample(kind, whole_frame(), DUMP_BYTES // len(kinds)))
        ms_total = ev0.elapsed_time(ev1)
        launches = pipe.launch_count() - launches0
        clocks = None   # the sampler keeps running through this output kind's e2e arm (see the end of measure)
        t = torch.tensor([ms_total], device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_step = float(t.item()) / args.steps
        value = W * H / (ms_step * 1e-3) / 1e6

        res = {"value": value, "ms_per_step": ms_step, "launches": int(launches), "clocks": clocks,
               "gather_mode": gather_mode}
        # per-kernel times (separate pass, CUDA events inside the library on the same stream)
        pipe.set_output_replicas([], 0)   # per-kernel times and the e2e arm run without the gather
        if world > 1:
            my_out = torch.empty((max_rows, W, 3), dtype=tdtype, device="cuda")
        pipe.set_profiling(True)
        ktimes = {"plan": [], "idct8": [], "idct_mid": [], "idct_large": [], "filter": []}
        for _ in range(max(5, min(args.steps, 20))):
            pipe.render_device(my_out.data_ptr(), row_bytes, stream.cuda_stream)
            for k, v in pipe.kernel_times_ms().items():
                ktimes[k].append(v)
        pipe.set_profiling(False)
        res["kernel_ms"] = {k: float(np.mean(v)) for k, v in ktimes.items()}

        # correctness spot check of the timed output against the reference decoder's pixels
        parity = None
        if fr.get("decoded") is None and rank == 0 and full and kind == "f32":
            # no cached pixels of the reference decoder: compare with the reference's own hot path (big frames)
            # or, for synthetic coefficient frames, with the C oracle on the first 512 rows
            got = whole_frame()
            from oracle import ref
            if fr.get("jxl") is not None and ref.available():
                frame = ref.Frame(fr["jxl"], host_cpu_info()["cores"])
                planar, _ = frame.render(-1)
                frame.close()
                want = np.moveaxis(planar, 0, 2)
                d = np.abs(got - want[:got.shape[0]])
                parity = {"peak_abs_err_vs_reference_hot_path": float(d.max()), "rows_checked": int(got.shape[0])}
                del planar, want, d
            else:
                from oracle import cpu as ocpu
                import copy
                sub = copy.copy(desc)
                rows = min(512, H)
                sub.ysize = rows
                for name_ in ("ac_strategy", "raw_quant", "epf_sharpness"):
                    setattr(sub, name_, getattr(desc, name_)[:rows // 8])
                sub.dc = desc.dc[:, :rows // 8]
                sub.ytox, sub.ytob = desc.ytox[:(rows // 8 + 7) // 8], desc.ytob[:(rows // 8 + 7) // 8]
                sub.band_y0_groups = sub.band_ny_groups = 0
                ng = sub.num_groups
                want = ocpu.render_frame(sub, coeffs[:, :ng], rcp_mode=0)
                halo = 8   # rows next to the cut see different neighbours
                parity = {"bit_exact_vs_oracle": bool(np.array_equal(got[:rows - halo], want[:rows - halo])),
                          "rows_checked": int(rows - halo)}
        if fr.get("decoded") is not None and rank == 0 and full:
            got = whole_frame()
            if kind == "f32":
                want = fr["decoded"][:got.shape[0]]
                d = np.abs(got - want)
                parity = {"peak_abs_err_vs_reference": float(d.max()),
                          "rmse_vs_reference": float(np.sqrt(np.mean(d * d))), "rows_checked": int(got.shape[0])}
            else:
                from oracle import ref
                if ref.available() and fr.get("jxl") is not None:
                    frame = ref.Frame(fr["jxl"], os.cpu_count() or 1)
                    want, _ = frame.render_out(-33, 2)        # the reference's own 8-bit sRGB bytes
                    frame.close()
                    d = np.abs(got.astype(np.int16) - want[:got.shape[0]].astype(np.int16))
                    parity = {"max_code_diff_vs_reference": int(d.max()),
                              "fraction_differing": float((d != 0).mean()), "rows_checked": int(got.shape[0])}
        res["parity"] = parity
        del gathered, my_out
        if world > 1 and os.environ.get("BENCH_KEEP_SYMM") != "1":
            # the host-fed arm has no gather: release the symmetric-memory frame buffers (and their peer mappings)
            import gc
            flat = None   # noqa: F841
            hdl = None
            gc.collect()
            torch.cuda.empty_cache()

        # ---------------- end-to-end arm: host buffers through the C ABI ----------------
        pipe.set_device_coefficients(None)
        # Host layout: one pinned [3][65536] block per AC group (what a pinned ACImage subclass gives
        # libjxl's entropy decoder to write into) -> each group is one DMA.
        if "host_groups" not in shared:
            host_all = pipeline.pinned_array((len(need), 3, abi.GROUP_COEFFS), coeffs.dtype)
            host_groups = {}
            h2d = 0
            for i, g in enumerate(need):
                n = desc.group_ncoeff(g)
                host_all[i] = coeffs[:, g]
                host_groups[g] = [host_all[i, c, :n] for c in range(3)]
                h2d += (2 * abi.GROUP_COEFFS + n) * coeffs.dtype.itemsize
            yb, xb = desc.ysize_blocks, desc.xsize_blocks
            h2d += yb * xb * (1 + 4 + 1 + 12) + desc.dequant.nbytes + 2 * desc.ytox.size
            shared["host_groups"], shared["h2d"] = host_groups, h2d
        host_groups, h2d = shared["host_groups"], shared["h2d"]
        host_out = pipeline.pinned_array((band_rows, W, 3), ndtype)
        d2h = host_out.nbytes

        from concurrent.futures import ThreadPoolExecutor
        if "pool" not in shared:
            shared["pool"] = ThreadPoolExecutor(n_submit_threads)
        pool = shared["pool"]

        # what libjxl's worker threads do after entropy-decoding their groups (dec_frame.cc:707-730);
        # the argument arrays are marshalled once, outside the timed region (ctypes overhead is not
        # part of the path)
        # each thread hands over whole AC-group rows (30 adjacent blocks at 8K -> one 23.6 MB DMA)
        xg = desc.xsize_groups
        rows_of = sorted({g // xg for g in need})
        batches = [pipe.make_batch([g for r in rows_of[tid::n_submit_threads] for g in need if g // xg == r], host_groups)
                   for tid in range(n_submit_threads)]

        # sparse hand-off: one batch (= one DMA of non-zero lists) per AC-group row
        if "sparse_batches" not in shared:
            sb = [[pipe.make_sparse_batch([g for g in need if g // xg == r], coeffs) for r in rows_of[tid::n_submit_threads]]
                  for tid in range(n_submit_threads)]
            shared["sparse_batches"] = sb
            shared["h2d_sparse"] = sum(b[3] for per in sb for b in per) + (shared["h2d"] - sum(
                (2 * abi.GROUP_COEFFS + desc.group_ncoeff(g)) * coeffs.dtype.itemsize for g in need))

        def run_e2e(mode: str) -> dict:
            def submit_slice(tid):
                if mode == "sparse":
                    for b in shared["sparse_batches"][tid]:
                        pipe.submit_sparse_batch(b, tid)
                else:
                    pipe.submit_batch(batches[tid], tid)

            phase = [0.0, 0.0, 0.0]

            def e2e_step():
                t0 = time.perf_counter()
                pipe.frame_begin(desc)
                pipe.frame_set_output(host_out)          # rows stream back as they finish
                t1 = time.perf_counter()
                list(pool.map(submit_slice, range(n_submit_threads)))
                t2 = time.perf_counter()
                pipe.frame_finish(host_out)
                t3 = time.perf_counter()
                phase[0] += t1 - t0
                phase[1] += t2 - t1
                phase[2] += t3 - t2

            for _ in range(2):
                e2e_step()
            barrier()
            phase[:] = [0.0, 0.0, 0.0]
            n_e2e = max(3, min(args.steps, 10))
            t0 = time.perf_counter()
            for _ in range(n_e2e):
                e2e_step()
            barrier()
            e2e_s = (time.perf_counter() - t0) / n_e2e
            log(f"[{kind}/{mode}] e2e phases (ms): begin {1e3 * phase[0] / n_e2e:.2f} "
                f"submit {1e3 * phase[1] / n_e2e:.2f} finish {1e3 * phase[2] / n_e2e:.2f}")
            te = torch.tensor([e2e_s], device="cuda")
            if world > 1:
                dist.all_reduce(te, op=dist.ReduceOp.MAX)
            h2d_t = torch.tensor([float(shared["h2d_sparse"] if mode == "sparse" else h2d), float(d2h)], device="cuda")
            if world > 1:
                dist.all_reduce(h2d_t)
            return {"value": W * H / float(te.item()) / 1e6, "unit": "Mpixel/s",
                    "h2d_bytes_per_step": int(h2d_t[0].item()), "d2h_bytes_per_step": int(h2d_t[1].item()),
                    "steps": n_e2e, "submit": mode}

        res["e2e"] = run_e2e(args.submit)
        # nvidia-smi samples (every 100 ms) from the start of the device-timed region to here: the timed
        # region alone lasts only K x 0.8 ms
        res["clocks"] = sampler.stop() if rank == 0 else None
        if res["clocks"] is not None:
            res["clocks"]["window"] = "device-timed region + per-kernel pass + e2e arm of this output kind"
        if not args.no_variants:
            res["e2e_other_submit"] = run_e2e("dense" if args.submit == "sparse" else "sparse")
        return res

    shared = {}
    dumps = {}
    other_kind = "srgb8" if args.output == "f32" else "f32"
    kinds = [args.output] if args.no_variants else [args.output, other_kind]
    pipeline.pin_side_info(desc)   # side info in page-locked memory, as the coefficient blocks are
    primary = measure(args.output, True)
    variant = None if args.no_variants else measure(other_kind, True)
    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name_, a in dumps.items():
            np.save(os.path.join(args.dump_outputs, f"{name_}.npy"), a)
    desc.out_format = abi.OUT_RGB_F32 if args.output == "f32" else abi.OUT_RGB_U8
    value, ms_step, launches, clocks = primary["value"], primary["ms_per_step"], primary["launches"], primary["clocks"]
    kavg, parity, gather_mode = primary["kernel_ms"], primary["parity"], primary["gather_mode"]
    pipe.close()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    # ---------------- roofline + CPU baseline (rank 0) ----------------
    peaks_path = ROOT / "MEASURED_PEAKS.json"
    if peaks_path.exists():
        peak = float(json.loads(peaks_path.read_text())["hbm_gbs"])
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    ab = algorithmic_bytes(desc, band_rows, 12 if args.output == "f32" else 3)
    k_idct = kavg["idct8"] + kavg["idct_mid"] + kavg["idct_large"]
    dominant = "filter" if kavg["filter"] >= k_idct else "idct"
    dom_ms = kavg["filter"] if dominant == "filter" else k_idct
    achieved = ab[dominant] / (dom_ms * 1e-3) / 1e9
    traffic, traffic_src = None, None
    try:   # DRAM bytes of the dominant kernel from the committed ncu capture of this workload, if there is one
        t = json.loads((ROOT / "profiles" / "ncu_traffic.json").read_text())[args.workload][args.output][dominant]
        if world == 1:
            traffic, traffic_src = float(t["bytes"]), t["capture"]
    except Exception:  # noqa: BLE001
        pass
    roofline = {"bound": "hbm", "kernel": "filter_strip_kernel" if dominant == "filter" else "idct8_tma_kernel+idct_mid_kernel+idct_large_kernel",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": peak_src, "algorithmic_bytes_per_launch": ab[dominant],
                "limiter": "instruction issue + shared-memory wavefronts, not HBM: the bit-exact arithmetic of an 8K step is "
                           "~0.33 ms of issue slots at 100% against 0.12 ms of HBM time (DESIGN.md §4, ncu summaries in profiles/)",
                "kernel_ms": kavg,
                "pipeline": {"algorithmic_bytes": ab["fused_path"],
                             "achieved_gbs": ab["fused_path"] / (sum(kavg.values()) * 1e-3) / 1e9,
                             "frac": ab["fused_path"] / (sum(kavg.values()) * 1e-3) / 1e9 / peak}}

    cpu_baseline = None
    if not args.no_cpu_baseline and world == 1 and fr.get("jxl") is not None:
        from oracle import ref
        cpu = host_cpu_info()
        cores = cpu["cores"]
        reps = 6
        nums = cpu_reference_numbers(fr, W, H, args.output, reps, [cores] if cores == 1 else [cores, 1])
        hot_by_kind = nums["hot"][cores]
        cpu_baseline = {"value": hot_by_kind[args.output], "unit": "Mpixel/s", "cores": cores, "kind": "reference",
                        "host": cpu, "hwy_target": ref.hwy_target(),
                        "sample": f"{reps} passes (+1 untimed first) of the reference's own hot-path code over the same "
                                  f"{W}x{H} frame (coefficients pre-decoded), geomean excluding the first "
                                  "(tools/speed_stats.cc:37-57); one_thread = the same with 1 thread (3 passes); "
                                  "full_decode = whole libjxl decoder incl. entropy decode",
                        "one_thread_mpixels_per_s": nums["hot"][1][args.output],
                        "full_decode_mpixels_per_s": nums["full"][cores],
                        "full_decode_one_thread_mpixels_per_s": nums["full"][1], "by_output": hot_by_kind}

    # ---------------- T_e2e: .jxl bytes -> pixels through the public JxlDecoder API ----------------
    # the reference with the jxl_b200 backend compiled in (oracle/build_ref.py "gpu" variant: build-time patched
    # dec_frame.cc / dec_group.cc + integration/libjxl_gpu_backend.h) against the stock decoder; the host
    # still does header parsing + ANS entropy decoding, the GPU does the transform path (SURVEY §8d scope 3)
    t_e2e = None
    if not args.no_cpu_baseline and world == 1 and fr.get("jxl") is not None:
        from oracle import ref
        if ref.available("gpu"):
            cpu = host_cpu_info()
            cores = cpu["cores"]
            try:
                ref.use_variant("gpu")
                runner = ref.Runner(cores)
                out_px = pipeline.pinned_array((H, W, 3), np.float32)   # the application's buffer (page-locked)
                by_mode = {}
                for mode in ("sparse", "dense"):
                    os.environ["JXLB_GPU_SPARSE"] = "1" if mode == "sparse" else "0"
                    before = ref.gpu_frames_taken()
                    ts = []
                    for _ in range(5):
                        t0 = time.perf_counter()
                        ref.decode_linear_f32(fr["jxl"], cores, out_px, runner)
                        ts.append(time.perf_counter() - t0)
                    taken = ref.gpu_frames_taken() - before
                    err = float(np.abs(out_px - fr["decoded"]).max()) if fr.get("decoded") is not None else None
                    by_mode[mode] = {"value": geomean_excluding_first(ts, W * H), "frames_on_gpu": int(taken),
                                     "peak_abs_err_vs_stock_decoder": err}
                os.environ.pop("JXLB_GPU_SPARSE", None)
                runner.close()
                t_e2e = {"value": by_mode["sparse"]["value"], "unit": "Mpixel/s", "threads": cores, "reps": 4,
                         "hand_off": by_mode,
                         "what": ".jxl codestream -> linear RGB f32 in a page-locked application buffer, public JxlDecoder "
                                 "API + JxlThreadParallelRunner; the patched FrameDecoder (oracle/_ref 'gpu' variant) entropy-decodes "
                                 "on the host and hands AC groups to libjxl_b200.so: sparse = non-zero lists appended by the patched "
                                 "DecodeACVarBlock, dense = pinned ACImage blocks",
                         "stock_decoder_mpixels_per_s": (cpu_baseline or {}).get("full_decode_mpixels_per_s"),
                         "stock_decoder_one_thread_mpixels_per_s": (cpu_baseline or {}).get("full_decode_one_thread_mpixels_per_s")}
            except Exception as e:  # noqa: BLE001
                t_e2e = {"error": repr(e)}
            finally:
                ref.use_variant("default")

    w_, h_, dist_, effort_, _, _, _ = WORKLOADS[args.workload]
    line = {
        "metric": "decode_mpixels_per_s", "value": value, "unit": "Mpixel/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_text(args.workload, desc, source, args.output),
                   "groups": desc.num_groups, "parallelism": f"band-sharded x{world}; all-gather: {gather_mode}" if world > 1 else "1 GPU",
                   "strategy_histogram": fr["hist"], "bpp": fr["bpp"],
                   "l2": "inputs larger than L2 (coefficients + XYB planes + output >> 126 MB per step)"},
        "e2e": {**primary["e2e"],
                "how": (f"frame_begin + frame_set_output + submit_groups (one AC-group row per call, {n_submit_threads} host "
                        "threads, pinned [group][3][65536] host blocks) + frame_finish; H2D / kernels / D2H overlap per row")
                if args.submit == "dense" else
                       (f"frame_begin + frame_set_output + submit_groups_sparse (one AC-group row per call, {n_submit_threads} "
                        "host threads, pinned non-zero lists as the entropy decoder would append them; zero-fill + "
                        "scatter kernel on the device) + frame_finish; H2D / kernels / D2H overlap per batch of rows")},
        "gpu_launches": int(launches), "roofline": roofline, "clocks": clocks, "parity": parity,
    }
    if cpu_baseline:
        line["cpu_baseline"] = cpu_baseline
    if t_e2e:
        line["t_e2e_decoder"] = t_e2e
    if variant is not None:
        # the same frame with the other output kind (same kernels; only the fused store differs)
        line["variants"] = {other_kind: {"output": OUTPUT_TEXT[other_kind], "value": variant["value"],
                                         "ms_per_step": variant["ms_per_step"], "kernel_ms": variant["kernel_ms"],
                                         "e2e": variant["e2e"], "e2e_other_submit": variant.get("e2e_other_submit"),
                                         "parity": variant["parity"],
                                         "cpu_reference_hot_path": (cpu_baseline or {}).get("by_output", {}).get(other_kind)},
                            "e2e_other_submit": primary.get("e2e_other_submit")}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
