#!/usr/bin/env python3
"""bench.py — headline benchmark of the conversion path (contract in the task statement).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload ...] [--layout ...] [--dump-outputs DIR]

A "step" = one ConversionPass::execute over the workload: BASELINE.json configs[1] — the SciFiHelmet stand-in
(seeded displaced sphere, 70 074 triangles, 3 x 2048^2 RGBA8 maps; the Khronos asset is not available offline) at
density 512.  Metric: Mgaussians/s.

  value      device-resident: scene already in HBM, CUDA events on the launching stream around the two kernel
             launches only, L2 flushed (256 MiB memset, untimed) before every timed step
  e2e        the same metric through the C ABI with HOST buffers.  N = 1: m2s_convert_host (pinned triangle + texture
             upload, GPU mip generation, convert, download of the records: a five-stream pipeline over triangle
             chunks, DESIGN.md section 4).  N > 1: every rank uploads ITS triangle
             shard (+ the maps the layout samples) over its own PCIe link, converts it, and downloads its records into
             its slice of ONE shared pinned host buffer (offsets from an all-gather of the counts) — the consumer of
             the reference's exportPly is a host vector (SceneManager.cpp:651-678), so no GPU-to-GPU traffic at all.
  roofline   algorithmic bytes (SURVEY 8d: N*B_out + T*144 + sum_maps min(4N, 4WH)) / live kernel time against the
             MEASURED HBM copy bandwidth in MEASURED_PEAKS.json; launch_shares = the two kernels timed live, separately
             (m2s_convert_timed: an event between them, no programmatic dependent launch)
  cpu_baseline / --impl reference
             the CPU restatement (oracle/, OpenMP, calibrated thread count) on the same workload and the same maps —
             the reference itself is an OpenGL 4.6 + Win32 GUI program and cannot be built or run here (no GL
             implementation on the box: profiles/r02_gl_probe.log), so kind = "port".
N > 1 (torchrun, one rank per GPU), device-resident leg: "every rank ends up holding all gaussians" (north_star's
all-gather).  Two strategies, both measured, the faster one (shard.choose_strategy on live timings) is `value`:
  replicate  every rank converts the whole scene itself — no traffic (wins when the records outweigh the work)
  shard      contiguous triangle ranges (shard.plan_work) + the fused gather: the fragment kernel stores each
             record span into every rank's final buffer over NVLink (m2s_convert_gather_enqueue)
The gathered buffer is verified (untimed) to be the single-GPU multiset on every rank: "gather_parity".
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from mesh2splat_b200 import _abi, synth  # noqa: E402

WORKLOAD_DEFAULT = "helmet_standin"  # BASELINE.json configs[1] (SciFiHelmet.glb stand-in)
# workload -> (scene factory, BASELINE density); only the default is the judged bench line
WORKLOADS = {"helmet_standin": (lambda: synth.helmet_standin(2048), 512),
             "sphere_1m": (lambda: synth.sphere_1m(2048), 256),
             "sponza_standin": (lambda: synth.sponza_standin(1024), 1024),
             "damaged_helmet_standin": (lambda: synth.damaged_helmet_standin(2048), 512)}
UNIT = "Mgaussians/s"
LAYOUTS = {"packed56": _abi.LAYOUT_PACKED56, "ref96": _abi.LAYOUT_REF96}
FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback
NVLINK_GBS = 770.0         # measured peer-copy bandwidth per direction (B200_PROFILING.md)


def _workload(args):
    make, dens = WORKLOADS[args.workload]
    return make(), (args.density or dens)


def maps_used(scene, layout: int) -> set:
    used = set()
    for p in scene.primitives:
        ids = [p.albedo_texture] if layout == _abi.LAYOUT_PACKED56 else \
            [p.albedo_texture, p.normal_texture, p.metallic_roughness_texture]
        used.update(i for i in ids if i >= 0)
    return used


def algorithmic_bytes(scene, n_gaussians: int, layout: int, n_triangles: int | None = None) -> int:
    """SURVEY 8(d) / BASELINE.md: N*B_out + T*144 + sum over maps the layout consumes of min(4N, 4WH)."""
    t = scene.triangle_count if n_triangles is None else n_triangles
    tex = sum(min(4 * n_gaussians, scene.textures[i].nbytes) for i in maps_used(scene, layout))
    return n_gaussians * _abi.STRIDES[layout] + t * 144 + tex


def make_config(args, scene, density: int, n_gaussians: int, world: int) -> dict:
    """The SAME dictionary in both arms (ours / --impl reference) for the same command line."""
    layout = LAYOUTS[args.layout]
    sizes = sorted({t.shape[0] for t in scene.textures})
    return {"workload": args.workload, "density": density, "layout": args.layout, "record_bytes": _abi.STRIDES[layout],
            "triangles": scene.triangle_count, "primitives": len(scene.primitives), "gaussians": n_gaussians,
            "textures": f"{len(scene.textures)} x RGBA8 {'/'.join(str(s) for s in sizes)}^2 (+ mips 1..4)",
            "maps_sampled": len(maps_used(scene, layout)),
            "l2": "GPU arm: flushed between iterations (256 MiB memset, untimed); CPU arm: not applicable",
            "gpus": world}


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:  # noqa: BLE001
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def profiled_traffic(layout_name: str):
    """dram bytes per step from the COMMITTED ncu capture (profiles/traffic.json) — not measured in this run."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f).get(layout_name)
    except Exception:  # noqa: BLE001
        return None


class ClockSampler:
    """Samples SM clock + throttle reasons of one GPU from a background thread (NVML, ~1 ms period)
    while the timed region runs; falls back to one nvidia-smi query if NVML is unavailable."""

    def __init__(self, index: int):
        import threading
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()
        except Exception:  # noqa: BLE001
            self._nv = None

    def _run(self):
        nv = self._nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons")
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
                r = int(get_reasons(self._h))
                for n, bit in names.items():
                    if r & bit:
                        self.reasons.add(n)
            except Exception:  # noqa: BLE001
                break
            time.sleep(0.001)

    def stop(self) -> dict:
        self._stop.set()
        if self._thr is not None:
            self._thr.join(timeout=2)
        if self._nv is None or not self.samples:
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", "--query-gpu=clocks.sm,clocks.max.sm",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=10).stdout
                a, b = [float(x) for x in out.strip().split(",")[:2]]
                return {"sm_mhz": a, "sm_max_mhz": b, "reasons": [], "samples": 1, "source": "nvidia-smi (after the timed region)"}
            except Exception:  # noqa: BLE001
                return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock query unavailable"], "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples), "source": "NVML, sampled during the timed region"}


def pin_array(a, torch, keep):
    t = torch.empty(a.nbytes, dtype=torch.uint8).pin_memory()
    v = t.numpy().view(a.dtype).reshape(a.shape)
    v[...] = a
    keep.append(t)
    return v


def pinned_scene(scene, torch, layout: int | None = None, tri_range=None):
    """The scene's arrays in pinned host memory (what a caller doing H2D every step holds).  tri_range = (first, count)
    keeps only that triangle range (multi-GPU shards: primitive ranges are clipped, bboxes kept); layout drops the
    maps the layout does not sample."""
    keep = []
    s = _abi.Scene.__new__(_abi.Scene)
    used = sorted(maps_used(scene, layout)) if layout is not None else list(range(len(scene.textures)))
    remap = {old: new for new, old in enumerate(used)}
    lo, n = tri_range if tri_range is not None else (0, scene.triangle_count)
    s.triangles = pin_array(scene.triangles[lo:lo + n], torch, keep)
    s.primitives = []
    for p in scene.primitives:
        a, b = max(p.first_triangle, lo), min(p.first_triangle + p.triangle_count, lo + n)
        s.primitives.append(_abi.Primitive(max(0, a - lo), max(0, b - a), p.base_color_factor, remap.get(p.albedo_texture, -1),
                                           remap.get(p.normal_texture, -1), remap.get(p.metallic_roughness_texture, -1),
                                           p.bbox_min, p.bbox_max))
    s.textures = [pin_array(scene.textures[i], torch, keep) for i in used]
    return s, keep


def cpu_convert_timed(scene, density, layout, reps: int, warm: int = 1):
    """The CPU port on the calibrated thread count: (gaussians, per-step seconds list, threads)."""
    import oracle
    prep = oracle.Prepared(scene)
    # torchrun exports OMP_NUM_THREADS=1, and more threads than usable cores is far slower than fewer
    # (128 allowed / 64 usable ran 30x slower at 128): time the candidates, keep the fastest
    cores = oracle.calibrate_threads(prep)
    out, n = None, 0
    for _ in range(max(1, warm)):
        n, _, out = prep.convert(density, layout, out=out, threads=cores)
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        n, _, out = prep.convert(density, layout, out=out, threads=cores)
        ts.append(time.perf_counter() - t0)
    return n, ts, cores


CPU_NOTE = ("CPU restatement of the reference shaders + GL-spec raster/sampler (oracle/), OpenMP, thread count calibrated; "
            "samples the same maps as the GPU arm; the reference's OpenGL path cannot run here (no GL implementation on the "
            "box: profiles/r02_gl_probe.log; Win32-only build)")


# ---------------------------------------------------------------------------------------------
def run_reference(args):
    """--impl reference: the CPU implementation of the path, all usable host cores, same workload/config."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    scene, density = _workload(args)
    layout = LAYOUTS[args.layout]
    steps = max(1, args.steps)
    n, ts, cores = cpu_convert_timed(scene, density, layout, steps, warm=max(1, min(args.warmup, 2)))
    dt = float(np.median(ts))
    val = n / dt / 1e6
    sample = (f"full workload ({scene.triangle_count} triangles -> {n} gaussians) per step; value = median of {steps} timed steps "
              f"(min {min(ts) * 1e3:.2f} ms, max {max(ts) * 1e3:.2f} ms)")
    line = {"impl": "reference", "metric": f"Mgaussians/s at density {density}", "value": val, "unit": UNIT, "n_gpus": world,
            "steps": steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": make_config(args, scene, density, n, world),
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample, "note": CPU_NOTE},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


DUMP_BYTES = 64_000_000


def dump_records(path: str, records: np.ndarray) -> None:
    """--dump-outputs: the records of the last timed step (structured, _abi.record_dtype), one DIR/<field>.npy per record
    field (one row per gaussian), and their count as DIR/total.npy.
    The kernels append records in atomic arrival order, which differs from run to run, so rows are sorted by their
    values (position first; the float bits mapped to integers that order like the floats, so -0.0 and NaN sort too).
    PACKED56 stores opacity as logit(alpha), +inf for an opaque gaussian (as the reference's .ply writer does); it is
    written as alpha.npy = sigmoid(opacity) in float64, finite and the form the parity tests compare it in.
    Beyond DUMP_BYTES a fixed seeded sample of the sorted rows is kept."""
    os.makedirs(path, exist_ok=True)
    bits = records.view(np.int32).reshape(len(records), -1)
    order = np.lexsort((bits ^ ((bits >> 31) & 0x7FFFFFFF)).T[::-1])
    rows = records[order]
    fields = {}
    for name in rows.dtype.names:
        if name == "opacity":
            with np.errstate(over="ignore"):
                fields["alpha"] = 1.0 / (1.0 + np.exp(-rows[name].astype(np.float64)))
        else:
            fields[name] = np.ascontiguousarray(rows[name])
    row_bytes = sum(a.nbytes // max(1, len(a)) for a in fields.values())
    keep = (DUMP_BYTES - 4096 * (len(fields) + 1)) // row_bytes
    if len(rows) > keep:
        pick = np.sort(np.random.default_rng(0).choice(len(rows), keep, replace=False))
        fields = {k: v[pick] for k, v in fields.items()}
    for name, a in fields.items():
        np.save(os.path.join(path, f"{name}.npy"), a)
    np.save(os.path.join(path, "total.npy"), np.array([len(records)], np.float64))


def record_hashes(buf, n: int, stride: int, torch):
    """Order-independent fingerprint of n records: sorted per-record 64-bit hashes (device tensor)."""
    w = buf[: n * stride].view(torch.int32).view(n, stride // 4).to(torch.int64)
    mult = torch.arange(1, stride // 4 + 1, device=buf.device, dtype=torch.int64) * 0x9E3779B1 + 0x7F4A7C15
    h = (w * mult).sum(dim=1)
    h = h ^ (h >> 29)
    return torch.sort(h).values


def run_ours(args):
    import torch
    import torch.distributed as dist
    from mesh2splat_b200.api import Context
    from mesh2splat_b200.shard import choose_strategy, estimate_cost, plan_work

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    layout = LAYOUTS[args.layout]
    stride = _abi.STRIDES[layout]
    scene, density = _workload(args)
    ctx = Context(local)
    ds = ctx.upload(scene)
    T = scene.triangle_count
    cap_total = 6 * density * density * max(1, len(scene.primitives))
    cap_total = min(cap_total, 60_000_000)
    # a dedicated (non-default) stream: everything timed is enqueued on it and the events are recorded on it
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    full = _abi.make_params(density, layout, 0.65, 0, _abi.FLAG_UNCAPPED, 0, 0, 0, 0)
    out = torch.empty(cap_total * stride, dtype=torch.uint8, device=dev)
    d_total = torch.zeros(1, dtype=torch.int64, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def timed(fn, reps, pre=None):
        """median ms of fn() over reps, L2 flushed before each, CUDA events on `stream`."""
        ts = []
        for _ in range(reps):
            flush.zero_()
            if pre:
                pre()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            fn()
            b.record(stream)
            torch.cuda.synchronize(dev)
            ts.append(a.elapsed_time(b))
        return float(np.median(ts))

    def local_full():
        ctx.convert_enqueue(ds, full, out, cap_total, None, d_total, stream.cuda_stream)

    # ---- N > 1: choose the strategy on live numbers -------------------------------------------------
    strategy, pg, shard_params, alt = "single", None, None, None
    lo, cnt_ = 0, T
    if world > 1:
        from mesh2splat_b200.shard import PeerGather
        for _ in range(3):
            local_full()
        t_single_us = timed(local_full, 5) * 1e3
        n_single = int(d_total.item())
        cost = estimate_cost(scene.triangles, scene.primitives[0].bbox_min, scene.primitives[0].bbox_max, density)
        lo, cnt_, row0, row1 = plan_work(T, world, density, cost)[rank]  # triangle ranges, or row bands for huge triangles
        shard_params = _abi.make_params(density, layout, 0.65, 0, _abi.FLAG_UNCAPPED, lo, cnt_, row0, row1)
        pg = PeerGather(ctx, cap_total, stride, dist, torch)
        model = choose_strategy(t_single_us, n_single, stride, world)
        strategy = model if args.strategy == "auto" else args.strategy
        t = torch.tensor([1.0 if strategy == "shard" else 0.0], device=dev)
        dist.broadcast(t, 0)  # every rank runs what rank 0 chose
        strategy = "shard" if t.item() > 0.5 else "replicate"

    def step_shard():
        pg.convert_enqueue(ds, shard_params, stream.cuda_stream)

    def run_timed(fn, pre=None):
        for _ in range(args.warmup):
            flush.zero_()
            if pre:
                pre()
            fn()
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        for a, b in evs:
            flush.zero_()  # evict L2 (126 MB) — untimed
            if pre:
                pre()      # untimed device-side barrier: the ranks enter the timed step together (no host skew in it)
            a.record(stream)
            fn()
            b.record(stream)
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        ms = sum(a.elapsed_time(b) for a, b in evs) / args.steps
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    def last_step(buf, n):
        """rank 0, --dump-outputs: host copy of the records the last timed step wrote"""
        if not args.dump_outputs or rank != 0:
            return None
        return buf[: n * stride].cpu().numpy().view(_abi.record_dtype(layout))

    clocks = ClockSampler(local) if rank == 0 else None
    gather_parity = None
    if world == 1:
        ms = run_timed(local_full)
        n_all = n_local = int(d_total.item())
        dumped = last_step(out, n_all)
    else:
        ms_rep = run_timed(local_full)
        n_all = int(d_total.item())
        dumped = last_step(out, n_all) if strategy == "replicate" else None
        ms_shard = run_timed(step_shard, pre=pg.barrier)
        torch.cuda.synchronize(dev)
        if strategy == "shard":
            dumped = last_step(pg.final, int(pg.total.item()))
        # untimed: the gathered buffer is the single-GPU multiset, on every rank
        n_g = int(pg.total.item())
        local_full()
        torch.cuda.synchronize(dev)
        ok = n_g == int(d_total.item())
        if ok:
            ok = bool(torch.equal(record_hashes(pg.final, n_g, stride, torch), record_hashes(out, n_g, stride, torch)))
        t = torch.tensor([1.0 if ok else 0.0], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        gather_parity = bool(t.item() > 0.5)
        ms = ms_shard if strategy == "shard" else ms_rep
        alt = {"replicate_ms": ms_rep, "shard_fused_gather_ms": ms_shard,
               "model": {"t_single_us": t_single_us, "choice": model}}
        ctx.convert_enqueue(ds, shard_params, out, cap_total, None, d_total, stream.cuda_stream)  # this rank's share, for the roofline
        torch.cuda.synchronize(dev)
        n_local = int(d_total.item())
    clk = clocks.stop() if clocks else None

    # ---- e2e through the C ABI with host buffers ----------------------------------------------------
    e2e = None
    e2e_steps = max(3, min(args.steps, 10))
    if world == 1:
        pscene, keep = pinned_scene(scene, torch)
        cs = pscene.c_struct()
        h_out = torch.empty(cap_total * stride, dtype=torch.uint8).pin_memory()
        h_np = h_out.numpy()
        for _ in range(2):
            rec, _, res = ctx.convert_host(pscene, density, layout, flags=_abi.FLAG_UNCAPPED, capacity=cap_total, out=h_np, c_scene=cs)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            rec, _, res = ctx.convert_host(pscene, density, layout, flags=_abi.FLAG_UNCAPPED, capacity=cap_total, out=h_np, c_scene=cs)
        torch.cuda.synchronize(dev)
        e2e_dt = (time.perf_counter() - t0) / e2e_steps
        # m2s_convert_host uploads the triangles and only the maps the layout consumes
        h2d = scene.triangles.nbytes + sum(scene.textures[i].nbytes for i in maps_used(scene, layout))
        d2h = int(res.written) * stride + 8
        e2e = {"value": int(res.written) / e2e_dt / 1e6, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
               "ms_per_step": e2e_dt * 1e3, "api": "m2s_convert_host (pinned host buffers; upload + mip generation + convert + download)"}
        # scene-resident "density slider" (SURVEY 3.2): convert + download only
        h_t = torch.empty(cap_total * stride, dtype=torch.uint8).pin_memory()
        def slider():
            o = ctx.convert(ds, density, layout, flags=_abi.FLAG_UNCAPPED, capacity=cap_total, out=out)
            h_t[: o.written * stride].copy_(out[: o.written * stride], non_blocking=True)
            torch.cuda.synchronize(dev)
            return o.written
        slider()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            nw = slider()
        sdt = (time.perf_counter() - t0) / e2e_steps
        e2e["resident_scene"] = {"value": nw / sdt / 1e6, "ms_per_step": sdt * 1e3,
                                 "what": "scene already on the GPU: m2s_convert + download of the records (the density-slider path)"}
    else:
        e2e = multi_gpu_e2e(args, scene, density, layout, ctx, dist, torch, dev, rank, world, cap_total, e2e_steps, out)

    line = None
    if rank == 0:
        value = n_all / (ms * 1e-3) / 1e6
        peak, peak_src = measured_peak()
        # ---- roofline of the conversion kernels: this rank's share, timed live ----
        kparams = shard_params if (world > 1 and strategy == "shard") else full
        ntri_k = cnt_ if (world > 1 and strategy == "shard") else T
        def kernels():
            ctx.convert_enqueue(ds, kparams, out, cap_total, None, d_total, stream.cuda_stream)
        kernel_ms = ms if world == 1 else timed(kernels, 5)
        n_k = int(d_total.item()) if world > 1 else n_all
        alg = algorithmic_bytes(scene, n_k, layout, ntri_k)
        achieved = alg / (kernel_ms * 1e-3) / 1e9
        shares = []
        for _ in range(7):
            flush.zero_(); torch.cuda.synchronize(dev)
            shares.append(ctx.convert_timed(ds, kparams, out, cap_total))
        ra, fr = float(np.median([s[0] for s in shares])) * 1e3, float(np.median([s[1] for s in shares])) * 1e3
        roofline = {"bound": "hbm", "kernel": "m2s::raster_kernel + m2s::fragment_kernel (the whole step)", "achieved": achieved,
                    "peak": peak, "unit": "GB/s", "frac": achieved / peak, "algorithmic_bytes": alg, "kernel_ms": kernel_ms,
                    "peak_source": peak_src,
                    "traffic": profiled_traffic(args.layout) if args.workload == WORKLOAD_DEFAULT else None,
                    "traffic_source": "committed ncu --set full capture (profiles/traffic.json), NOT measured in this run",
                    "launch_shares": {"raster_kernel_us": round(ra, 2), "fragment_kernel_us": round(fr, 2),
                                      "raster_share": round(ra / (ra + fr), 3), "fragment_share": round(fr / (ra + fr), 3),
                                      "source": "measured in this run: m2s_convert_timed, CUDA event between the kernels, no PDL "
                                                "overlap, L2 flushed, median of 7"}}
        if world > 1:  # bytes that must cross NVLink per GPU for "every rank holds the full buffer" when sharded
            nv = (n_all - n_local) * stride
            roofline["nvlink"] = {"ingress_bytes_per_gpu": int(nv), "peak_GBps": NVLINK_GBS, "floor_ms": nv / (NVLINK_GBS * 1e9) * 1e3,
                                  "note": "sharded strategy only; measured peer-copy bandwidth per direction (B200_PROFILING.md)"}
        cpu = None
        if world == 1:  # bounded CPU sample on this box's host cores
            n, ts, cores = cpu_convert_timed(scene, density, layout, 5)
            cdt = float(np.median(ts))
            cpu = {"value": n / cdt / 1e6, "unit": UNIT, "cores": cores, "kind": "port",
                   "sample": f"full workload ({scene.triangle_count} triangles -> {n} gaussians), median of 5 timed steps after warm-up",
                   "note": CPU_NOTE}
        cfg = make_config(args, scene, density, n_all, world)
        parallelism = ("1 GPU" if world == 1 else
                       (f"{strategy}: " + ("triangle shards + fused gather (peer stores into every rank's final buffer over NVLink)"
                                           if strategy == "shard" else "every rank converts the whole scene (no traffic)")))
        line = {"metric": f"Mgaussians/s at density {density}", "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": cfg, "parallelism": parallelism, "e2e": e2e,
                "gpu_launches": 2 * args.steps,  # raster_kernel + fragment_kernel per timed step (no memsets: the scheduler re-arms itself)
                "clocks": clk, "roofline": roofline, "cpu_baseline": cpu}
        if world > 1:
            line["strategy"] = strategy
            line["strategies_measured"] = alt
            line["gather_parity"] = gather_parity
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    ds.free()
    ctx.close()
    if dumped is not None:
        dump_records(args.dump_outputs, dumped)
    if line is not None:
        print(json.dumps(line))


def multi_gpu_e2e(args, scene, density, layout, ctx, dist, torch, dev, rank, world, cap_total, steps, scratch_out):
    """Every rank: upload ITS triangle shard (+ the maps the layout samples) from pinned host memory, convert, download its
    records into its slice of ONE shared pinned host buffer.  Offsets = exclusive scan of the all-gathered counts.
    Timed on the host between barriers, max over ranks (the transfers are host<->device, there is no device-only clock)."""
    from multiprocessing import shared_memory
    from mesh2splat_b200.shard import plan_shards
    stride = _abi.STRIDES[layout]
    T = scene.triangle_count
    lo, cnt = plan_shards(T, world)[rank]
    pscene, keep = pinned_scene(scene, torch, layout)   # the whole scene in pinned host memory; each rank uploads its part
    cs = pscene.c_struct()
    nbytes = cap_total * stride
    name = f"m2s_bench_{os.environ.get('MASTER_PORT', '0')}"
    shm = None
    if rank == 0:
        try:
            shared_memory.SharedMemory(name=name).unlink()
        except Exception:  # noqa: BLE001
            pass
        shm = shared_memory.SharedMemory(name=name, create=True, size=nbytes)
    dist.barrier()
    if rank != 0:
        shm = shared_memory.SharedMemory(name=name)
    host = torch.frombuffer(shm.buf, dtype=torch.uint8, count=nbytes)
    rt = torch.cuda.cudart()
    reg = rt.cudaHostRegister(host.data_ptr(), nbytes, 0)
    pinned = int(reg) == 0 if not isinstance(reg, tuple) else int(reg[0]) == 0
    d_out = scratch_out
    counts = torch.zeros(world, dtype=torch.int64, device=dev)
    mine = torch.zeros(1, dtype=torch.int64, device=dev)
    h2d_box = [0]

    def step():
        # H2D: the shard's triangles + the texture rows they sample (m2s_scene_upload_range), GPU mip generation
        dsub = ctx.upload_range(pscene, layout, lo, cnt, c_scene=cs)
        h2d_box[0] = dsub.h2d_bytes()
        o = ctx.convert(dsub, density, layout, flags=_abi.FLAG_UNCAPPED, capacity=cap_total, out=d_out,
                        first_triangle=lo, triangle_count=cnt)
        mine.fill_(o.written)
        dist.all_gather_into_tensor(counts, mine)               # 8 bytes per rank
        c = counts.cpu()
        off = int(c[:rank].sum())
        n = int(o.written)
        if off + n <= cap_total and n:
            host[off * stride:(off + n) * stride].copy_(d_out[: n * stride], non_blocking=pinned)   # D2H into the shared buffer
        torch.cuda.synchronize(dev)
        dsub.free()
        return int(c.sum()), n

    for _ in range(2):
        step()
    dist.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        n_all, n_mine = step()
    torch.cuda.synchronize(dev)
    dt_local = (time.perf_counter() - t0) / steps
    t = torch.tensor([dt_local], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dt = float(t.item())
    tot = torch.tensor([float(h2d_box[0]), float(n_mine * stride)], dtype=torch.float64, device=dev)
    dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    # untimed check on rank 0: the shared host buffer is the single-GPU multiset
    dist.barrier()
    ok = None
    if rank == 0:
        ds_full = ctx.upload(scene)
        o = ctx.convert(ds_full, density, layout, flags=_abi.FLAG_UNCAPPED, capacity=cap_total)
        got = host[: n_all * stride].to(dev)
        ok = bool(o.written == n_all and torch.equal(record_hashes(got, n_all, stride, torch), record_hashes(o.data, n_all, stride, torch)))
        ds_full.free()
    dist.barrier()
    rt.cudaHostUnregister(host.data_ptr())
    del host
    shm.close()
    if rank == 0:
        shm.unlink()
    return {"value": n_all / dt / 1e6, "unit": UNIT, "h2d_bytes_per_step": int(tot[0].item()), "d2h_bytes_per_step": int(tot[1].item()),
            "ms_per_step": dt * 1e3, "host_buffer_parity": ok, "shared_buffer_pinned": bool(pinned),
            "api": f"{world} ranks x (m2s_scene_upload_range: the rank's triangle shard + the texture rows it samples; m2s_convert; download "
                   "into its slice of one shared pinned host buffer, offsets from an all-gather of the counts); host clock between "
                   "barriers, max over ranks"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--layout", default="packed56", choices=sorted(LAYOUTS))
    ap.add_argument("--workload", default=WORKLOAD_DEFAULT, choices=sorted(WORKLOADS),
                    help="default: BASELINE configs[1] stand-in; sphere_1m = configs[3] (the multi-GPU config)")
    ap.add_argument("--density", type=int, default=0, help="sampling density R (0 = the workload's BASELINE density)")
    ap.add_argument("--strategy", default="auto", choices=["auto", "shard", "replicate"],
                    help="N>1, device-resident leg: auto = shard.choose_strategy on live timings")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the records of the last timed step, sorted, as DIR/<field>.npy (PACKED56 opacity as alpha.npy) and their count as DIR/total.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU path's records (--impl ours)")
    args.warmup = max(3, args.warmup) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
