#!/usr/bin/env python
"""Benchmark of the tri-plane volume-rendering hot path: rendered rays/s (48+48 samples).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload c2]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

A step is one pass of the hot path over one batch of synthetic input (BASELINE.json configs[1] restricted
to the path: batch 8, 64^2 rays, 48+48 samples, disentangled decoder, two 3x32x256x256 plane sets):
    RaySampler -> plane statistics + normalisation -> channel-last staging -> coarse field -> coarse weights
    -> importance resampling -> fine field -> merge + composite            (+ NCCL all-gather of the images, N > 1)
`value` times that with the raw planes already resident in HBM; `e2e` times the same call sequence from
pinned HOST buffers (H2D of the planes and cameras, D2H of the rendered maps inside the timed region).
Multi-GPU is weak scaling: every rank renders its own batch of 8 (batch-first sharding, SURVEY.md §8e).

Other workloads (--workload): c1 (batch 1), c3 (batch 32, 128^2), c4 (training step, forward+backward), c5 (one identity under
64 poses, 256^2 rays, 96+96).  --cuda-graph replays the step as one CUDA graph (nerffaceediting_b200.graphs); the default run
reports that variant beside the eager numbers under "cuda_graph" (single GPU, inference workloads).

--impl reference times the CPU restatement of the reference path (oracle/, all host threads) on the same
workload, one batch item per step.  Prints ONE JSON line (rank 0).

--dump-outputs DIR writes what the timed step returned in its last step (rank 0: the rendered maps rgb, seg, depth, wsum; the
training step: its loss and the gradients it leaves on the planes and the decoder) as DIR/<name>.npy in float32.  The inputs are
seeded, so two builds run with the same arguments can be compared output for output.  With N > 1 the training step's decoder
gradients are rank 0's own: the step all-reduces a flattened copy of them and does not write the sum back.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (batch per GPU, neural resolution, coarse, fine)
    "c2": dict(batch=8, res=64, s_c=48, s_f=48, desc="configs[1] hot path: batch 8, 64^2 rays, 48+48, DisentangledOSGDecoder, 2 plane sets 3x32x256x256 fp32"),
    "c1": dict(batch=1, res=64, s_c=48, s_f=48, desc="configs[0]-shaped: batch 1, 64^2 rays, 48+48, DisentangledOSGDecoder"),
    "c3": dict(batch=32, res=128, s_c=48, s_f=48, desc="configs[2]-shaped: batch 32, 128^2 rays, 48+48"),
    "c4": dict(batch=32, res=64, s_c=48, s_f=48, train=True,
               desc="configs[3]-shaped training step: renderer forward+backward, batch 32/GPU, 64^2 rays, 48+48, gradients to planes + decoders"),
    # configs[4]: one identity (ONE plane set, batch-broadcast, SURVEY.md §8e) under 64 poses per GPU, 256^2 rays, 96+96 samples
    "c5": dict(batch=64, plane_batch=1, res=256, s_c=96, s_f=96,
               desc="configs[4]-shaped video sweep: 64 poses/GPU of one identity (plane batch 1, broadcast), 256^2 rays, 96+96"),
}
GATHER_BYTES_PER_SAMPLE_SET = 12 * 32 * 4      # 3 planes x 4 taps x 32 ch x fp32 (SURVEY.md §8d)
MLP_FLOP_PER_SAMPLE = 14336                    # DisentangledOSGDecoder (SURVEY.md §8d)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)", d
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)", {}


def tensor_frac(mlp_tflops, precision, peaks):
    """Tensor-pipe share of the decoder MLPs: the MMA work actually issued (bf16x3 runs every product as three bf16 MMAs) over the
    measured dense bf16 peak of MEASURED_PEAKS.json; None for the FFMA mode or when no measured peak is available."""
    try:
        peak = float(peaks.get("bf16_tflops") or 0.0)
    except (TypeError, ValueError, AttributeError):
        return None
    if precision == "fp32" or peak <= 0.0:
        return None
    return mlp_tflops * (3.0 if precision == "bf16x3" else 1.0) / peak


def bind_to_gpu_numa(torch, local):
    """Pin this process to the cores of the NUMA node its GPU hangs off BEFORE any pinned host memory is allocated (first-touch
    places the pages there), so that N ranks uploading at once do not all read one socket's memory (VERDICT r01 weak #7).
    Returns a description for the JSON line; a box that exposes a single node (or no topology) is left alone."""
    info = {"gpu_numa_node": None, "bound_cpus": None, "nodes": None}
    try:
        nodes = sorted(int(d[4:]) for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit())
        info["nodes"] = len(nodes)
        p = torch.cuda.get_device_properties(local)
        bdf = f"{getattr(p, 'pci_domain_id', 0):04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read().strip())
        info["gpu_numa_node"] = node
        if node >= 0 and len(nodes) > 1:
            cpus = set()
            for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
                lo, _, hi = part.partition("-")
                cpus.update(range(int(lo), int(hi or lo) + 1))
            allowed = cpus & os.sched_getaffinity(0)
            if allowed:
                os.sched_setaffinity(0, allowed)
                info["bound_cpus"] = len(allowed)
    except Exception as exc:    # noqa: BLE001
        info["error"] = f"{type(exc).__name__}: {exc}"[:160]
    return info


def measure_l2_gather(torch, _lib, device):
    """GB/s of random 128-byte-line gathers out of an L2-resident 25 MB table with the field kernel's access shape (LDG.128, 8 lanes
    per line): the roof the tri-plane gather runs under (SURVEY.md §8d asks for gather_bytes / BW_L2; nothing publishes BW_L2, so
    it is measured here, live, on the box the bench runs on).  Two launch shapes: the best one found by the sweep in
    profiles/l2_gather_r02.txt (32 warps x 8 loads in flight per SM) and the field kernel's own (8 gather warps x 12)."""
    import ctypes
    n_lines = 3 * 256 * 256
    table = torch.zeros(n_lines * 32, device=device)
    sink = torch.zeros(1, device=device)
    lib = _lib.load()
    lines = ctypes.c_int64(0)
    stream = torch.cuda.current_stream(device).cuda_stream
    out = {}
    for name, warps, depth in (("peak", 32, 8), ("kernel_shape", 8, 12)):
        iters = 6144 // depth
        best = None
        for rep in range(4):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            _lib.check(lib.nfe_bench_l2_gather(table.data_ptr(), n_lines, warps, depth, iters, ctypes.byref(lines), sink.data_ptr(), stream),
                       "nfe_bench_l2_gather")
            e1.record()
            e1.synchronize()
            ms = e0.elapsed_time(e1)
            if rep and (best is None or ms < best):       # the first launch warms the table into L2
                best = ms
        out[name] = lines.value * 128 / (best * 1e-3) / 1e9
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 100 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.file = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=self.file, stderr=subprocess.DEVNULL)
        except OSError:
            pass

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        self.proc.wait()
        self.file.flush()
        rows = [r.strip().split(", ") for r in open(self.file.name) if r.strip()]
        os.unlink(self.file.name)
        sm, mx, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.strip().lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_inputs(torch, wl, device, seed):
    import synth_inputs as synth
    from nerffaceediting_b200.triplane import DisentangledOSGDecoder
    g = torch.Generator(device="cpu").manual_seed(seed)
    n = wl["batch"]
    pb = wl.get("plane_batch", n)
    raw_host = torch.randn(pb, 96, 256, 256, generator=g).pin_memory() if device.type == "cuda" else torch.randn(pb, 96, 256, 256, generator=g)
    torch.manual_seed(seed)
    dec = DisentangledOSGDecoder(32, {'decoder_lr_mul': 1, 'decoder_output_dim': 32, 'decoder_seg_dim': 15})
    c2w, k = synth.camera_sweep(n)
    opts = dict(synth.FFHQ_RENDERING_OPTIONS, depth_resolution=wl["s_c"], depth_resolution_importance=wl["s_f"], nfe_deterministic=True)
    return raw_host, dec, c2w, k, opts


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, arrays, budget=DUMP_BYTES):
    """Write {name: tensor} as out_dir/<name>.npy in float32, at most `budget` bytes in all.  Arrays of up to 1 MB are stored
    whole; when the larger ones do not fit in the rest of the budget, each keeps the same fraction of its rows (last dimension
    whole; a vector's rows are its elements), picked with a fixed seed, so that two runs on the same shapes store the same
    elements."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    header = 128                                    # bytes of a .npy header for these shapes
    large = {n_ for n_, t in arrays.items() if t.numel() * 4 > (1 << 20)}
    room = budget - sum(header + (0 if n_ in large else t.numel() * 4) for n_, t in arrays.items())
    if room <= 0:
        raise ValueError(f"the arrays of up to 1 MB alone fill the {budget}-byte budget")
    total = sum(arrays[n_].numel() * 4 for n_ in large)
    for name, t in arrays.items():
        a = t.detach().float()
        if name in large and total > room:
            rows = a.reshape(-1, a.shape[-1] if a.dim() >= 2 else 1)
            keep = rows.shape[0] * room // total
            if keep == 0:                           # one row is wider than this array's share: sample elements instead
                rows = a.reshape(-1, 1)
                keep = rows.shape[0] * room // total
            idx = np.sort(np.random.default_rng(0).choice(rows.shape[0], keep, replace=False))
            a = rows[torch.from_numpy(idx).to(a.device)]
        np.save(os.path.join(out_dir, name + ".npy"), a.cpu().numpy())


def hot_path_step(torch, mods, raw, dec, c2w, k, res, opts):
    """The public-API call sequence of TriPlaneGenerator.synthesis restricted to the hot path
    (triplane.py:84,95,113-119)."""
    o, d = mods["sampler"](c2w, k, res)
    norm, mean, std = mods["normalize_plane"](raw)
    n, _, h, w = raw.shape
    planes = raw
    if mods.get("swap"):
        # appearance swap (BASELINE configs[2], triplane.py:93-107): every item is de-normalised with its neighbour's statistics
        planes = mods["denormalize_plane"](norm, mean.roll(1, 0), std.roll(1, 0))
    return mods["renderer"](norm.view(n, 3, 32, h, w), planes.view(n, 3, 32, h, w), dec, o, d, opts)


def cpu_reference_rate(torch, wl, steps, warmup, threads=None):
    """rays/s of the CPU restatement of the reference path (oracle/), one batch item per step."""
    import numpy as np
    import synth_inputs as synth
    from oracle import nfe_oracle as orc
    threads = threads or os.cpu_count() or 1
    os.environ["OMP_NUM_THREADS"] = str(threads)
    orc.set_num_threads(threads)        # torchrun exports OMP_NUM_THREADS=1 and libgomp has already read it
    raw_host, dec, c2w, k, opts = make_inputs(torch, dict(wl, batch=1, plane_batch=1), torch.device("cpu"), 0)
    raw = raw_host.numpy()
    kind, a, b, cd, sd = orc.decoder_nets(dec)
    rays = wl["res"] ** 2
    table = torch.linspace(opts['ray_start'], opts['ray_end'], wl["s_c"]).numpy()
    u = torch.linspace(0, 1, wl["s_f"]).numpy()

    def step():
        o, d = orc.generate_rays(c2w.numpy(), k.numpy(), wl["res"])
        norm, _, _ = orc.normalize_plane(raw)
        dc = orc.sample_stratified(1, rays, wl["s_c"], table=table, ray_start=opts['ray_start'], ray_end=opts['ray_end'])
        return orc.render(kind, a, b, norm.reshape(1, 3, 32, 256, 256), raw.reshape(1, 3, 32, 256, 256), o, d, dc, u, wl["s_f"], cd, sd)

    for _ in range(warmup):
        step()
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
    best, mean = min(times), sum(times) / len(times)
    return {"rays_per_s_best": rays / best, "rays_per_s_mean": rays / mean, "ms_per_step": mean * 1e3, "cores": threads,
            "sample": f"1 of {wl['batch']} batch items (poses) per step ({rays} rays, {wl['s_c']}+{wl['s_f']} samples, 2 plane sets, stats+normalise included), "
                      f"{steps} steps after {warmup} warm-up"}


def run_reference(args, wl):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_reference_rate(torch, wl, max(args.steps, 1), max(args.warmup, 1))
    line = {"impl": "reference", "metric": f"rendered rays/sec ({wl['s_c']}+{wl['s_f']} samples)", "value": r["rays_per_s_mean"], "unit": "rays/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl["desc"], "rays_per_gpu_per_step": wl["res"] ** 2, "sampling": "deterministic (parity mode)",
                       "parallelism": f"host CPU, {r['cores']} OpenMP threads (rank 0 only)",
                       "cache": "n/a (CPU arm)",
                       "sample": f"1 of the workload's {wl['batch']} batch items per step (a bounded sample of the same workload: rays/s is a rate, "
                                 "the per-item work is identical for every item)",
                       "note": "CPU restatement (oracle port) of the reference renderer on the box's host cores"},
            "cpu_baseline": {"value": r["rays_per_s_mean"], "unit": "rays/s", "cores": r["cores"], "kind": "port", "sample": r["sample"]},
            "e2e": {"value": r["rays_per_s_mean"], "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the extra measurements reported beside the contract's numbers "
                    "(unpatched-generator flow, stochastic sampling, configs[3] training step)")
    ap.add_argument("--two-gather", action="store_true",
                    help="disable the single-gather identity (gather both plane sets, as the reference does)")
    ap.add_argument("--precision", default="bf16x3", choices=["fp32", "bf16x3", "bf16"],
                    help="decoder MLP arithmetic (rendering_options['nfe_precision'])")
    ap.add_argument("--swap-statistics", action="store_true",
                    help="appearance swap inside the step (BASELINE configs[2]): denormalize_plane with the neighbouring item's mean/std "
                         "before the render (one more 3-pass-equivalent kernel over the planes; the single-gather identity still applies)")
    ap.add_argument("--cuda-graph", action="store_true",
                    help="replay the step as ONE CUDA graph (nerffaceediting_b200.graphs; single-GPU inference workloads; "
                         "pays off where the step is launch-bound, i.e. c1)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the timed step returned in its last step to DIR/<name>.npy (float32; a fixed sample of rows when "
                         f"the arrays exceed {DUMP_BYTES >> 20} MB)")
    args = ap.parse_args()
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        if args.dump_outputs:
            raise SystemExit("--dump-outputs writes the outputs of the CUDA path (--impl b200)")
        return run_reference(args, wl)

    import torch
    import torch.distributed as dist
    from nerffaceediting_b200 import _lib
    from nerffaceediting_b200.ray_sampler import RaySampler
    from nerffaceediting_b200.renderer import DisentangledImportanceRenderer
    from nerffaceediting_b200.triplane import denormalize_plane, normalize_plane

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback exists)"
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"          # keep NCCL's version banner off stdout: rank 0 prints ONE JSON line
        dist.init_process_group("nccl", device_id=device)
    steps, warmup = max(args.steps, 1), max(args.warmup, 3)
    numa = bind_to_gpu_numa(torch, local)
    mods = {"sampler": RaySampler(), "normalize_plane": normalize_plane, "denormalize_plane": denormalize_plane,
            "renderer": DisentangledImportanceRenderer(), "swap": bool(args.swap_statistics)}
    if args.swap_statistics and (wl.get("train") or wl["batch"] < 2):
        raise SystemExit("--swap-statistics needs an inference workload with at least two batch items")

    raw_host, dec, c2w_host, k_host, opts = make_inputs(torch, wl, device, 1000 + rank)
    opts["nfe_precision"] = args.precision
    opts["nfe_single_gather"] = not args.two_gather
    sets_gathered = 2 if (args.two_gather or args.precision == "fp32") else 1
    dtype = {"fp32": "f32", "bf16x3": "f32 (gather, compositing) + bf16x3 split tensor-core MLP with f32 accumulate",
             "bf16": "f32 (gather, compositing) + bf16 tensor-core MLP"}[args.precision]
    dec = dec.to(device)
    raw = raw_host.to(device)
    c2w, k = c2w_host.to(device), k_host.to(device)
    c2w_host, k_host = c2w_host.pin_memory(), k_host.pin_memory()
    n, res = wl["batch"], wl["res"]
    rays_per_rank = n * res * res
    # N > 1: the render goes through the product's sharding API (nerffaceediting_b200.sharding.ShardedRenderer, batch-first:
    # every rank renders its own items): deferred depth clamp, nfe_finish_depth, and the one data-path collective — the
    # all-gather of the packed [rgb|seg|depth|wsum] maps (SURVEY.md §8e) — on a communication stream out of a 2-deep ring, so
    # the gather of step i overlaps the render of step i+1
    from nerffaceediting_b200 import sharding
    sharded = sharding.ShardedRenderer(mods["renderer"], overlap=True) if world > 1 else None
    if sharded is not None:
        plain_renderer = mods["renderer"]
        mods["renderer"] = lambda norm_, planes_, dec_, o_, d_, opts_: sharded(norm_, planes_, dec_, o_, d_, opts_, local_batch=True)
    packed_ring = [torch.empty((n, res * res, 49), device=device) for _ in range(2)]
    ring = {"i": 0}

    def pack_local(rgb, seg, depth, wsum):
        slot = ring["i"] & 1
        ring["i"] += 1
        return torch.cat([rgb, seg, depth, wsum], dim=-1, out=packed_ring[slot])

    train = bool(wl.get("train"))
    if train:
        # training step (configs[3]): forward + backward of a fixed random projection of every output; gradients reach the raw
        # planes (through normalize_plane and the renderer) and the decoder parameters; data-parallel ranks all-reduce the
        # decoder gradients (the plane gradients belong to the per-item backbone activations and stay local)
        raw.requires_grad_(True)
        gw = torch.Generator(device="cpu").manual_seed(5)
        proj = [torch.randn(n, res * res, c, generator=gw).to(device) for c in (32, 15, 1, 1)]
        params = list(dec.parameters())

        def train_step(planes_dev, c2w_dev, k_dev):
            planes_dev.grad = None
            for p_ in params:
                p_.grad = None
            out = hot_path_step(torch, mods, planes_dev, dec, c2w_dev, k_dev, res, opts)
            loss = sum((o_ * w_).sum() for o_, w_ in zip(out, proj))
            loss.backward()
            if world > 1:
                flat = torch.cat([p_.grad.reshape(-1) for p_ in params])
                dist.all_reduce(flat)
            return loss

    graphed = None
    if args.cuda_graph:
        if train or world > 1:
            raise SystemExit("--cuda-graph covers the single-GPU inference workloads (the training step and the NCCL ring stay eager)")
        from nerffaceediting_b200 import graphs

    def step_resident():
        if train:
            return train_step(raw, c2w, k)
        if graphed is not None:
            return graphed["resident"]()
        with torch.no_grad():
            return hot_path_step(torch, mods, raw, dec, c2w, k, res, opts)      # N > 1: a sharding.PendingMaps (gather in flight)

    # ---- end to end from HOST buffers: every step uploads its planes + cameras from pinned memory and reads the maps back.
    # Uploads run on a side stream into a 2-deep device ring, so the copy of step i+1 overlaps the render of step i (what a
    # caller streaming frames would do); the host consumes the result of step i-1 while step i renders.
    out_host = [torch.empty((n, res * res, 49), dtype=torch.float32).pin_memory() for _ in range(2)]
    dev_in = [torch.empty_like(raw) for _ in range(2)]
    dev_cam = [(torch.empty_like(c2w), torch.empty_like(k)) for _ in range(2)]
    # the 201 MB of planes go up in batch-item chunks dealt over two copy streams (two DMA queues in flight per rank)
    copy_streams = [torch.cuda.Stream(device=device) for _ in range(2)]
    copy_stream = copy_streams[0]
    n_up = min(4, raw_host.shape[0])
    up_bounds = [raw_host.shape[0] * j // n_up for j in range(n_up + 1)]
    uploaded = [[torch.cuda.Event() for _ in range(2)] for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    done = [torch.cuda.Event() for _ in range(2)]
    e2e_state = {"i": 0}

    def upload(slot):
        for si, cs in enumerate(copy_streams):
            with torch.cuda.stream(cs):
                cs.wait_event(consumed[slot])                           # the render that last read this slot has finished
                for j in range(si, n_up, 2):
                    dev_in[slot][up_bounds[j]:up_bounds[j + 1]].copy_(raw_host[up_bounds[j]:up_bounds[j + 1]], non_blocking=True)
                if si == 0:
                    dev_cam[slot][0].copy_(c2w_host, non_blocking=True)
                    dev_cam[slot][1].copy_(k_host, non_blocking=True)
                uploaded[slot][si].record(cs)

    def h2d_rate_concurrent(reps=6):
        """GB/s of this rank's pinned-host -> device plane upload while EVERY rank uploads at once (a bandwidthTest of the box's
        host fabric under the bench's own traffic pattern); max over ranks of the time, so the slowest link counts."""
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            dev_in[0].copy_(raw_host, non_blocking=True)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=device, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return raw_host.numel() * 4 * reps / (ms * 1e-3) / 1e9

    loss_host = torch.empty((), dtype=torch.float32).pin_memory()

    def step_e2e():
        if train:
            # a training step fed from host memory: planes + cameras up, loss scalar back
            dev_in[0].requires_grad_(False).copy_(raw_host, non_blocking=True)
            dev_cam[0][0].copy_(c2w_host, non_blocking=True)
            dev_cam[0][1].copy_(k_host, non_blocking=True)
            loss = train_step(dev_in[0].requires_grad_(True), dev_cam[0][0], dev_cam[0][1])
            loss_host.copy_(loss.detach(), non_blocking=True)
            torch.cuda.current_stream().synchronize()
            return
        i = e2e_state["i"]
        slot = i & 1
        main = torch.cuda.current_stream()
        with torch.no_grad():
            if i == 0:
                consumed[0].record(main); consumed[1].record(main)
                upload(0)
            upload(slot ^ 1)                                            # next step's inputs, overlapping this step's render
            main.wait_event(uploaded[slot][0])
            main.wait_event(uploaded[slot][1])
            if graphed is not None and graphed["slot"] is not None:
                rgb, seg, depth, wsum = graphed["slot"][slot]()
                packed = pack_local(rgb, seg, depth, wsum)
            else:
                out = hot_path_step(torch, mods, dev_in[slot], dec, dev_cam[slot][0], dev_cam[slot][1], res, opts)
                packed = sharded.last_packed if sharded is not None else pack_local(*out)    # this rank's maps go back to ITS host
            consumed[slot].record(main)
            out_host[slot].copy_(packed, non_blocking=True)
            done[slot].record(main)
            if i > 0:
                done[slot ^ 1].synchronize()                            # the caller reads the previous step's result
        e2e_state["i"] = i + 1

    def timed(fn, with_stage_timer):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        if with_stage_timer:
            _lib.timing_read(reset=True)
            _lib.timing_enable(True)
        launches0 = _lib.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps - 1):
            fn()
        last = fn()         # outside the loop, so that no step runs while the previous step's outputs are still held
        if sharded is not None:
            sharded.drain()                                       # the last steps' all-gathers are inside the timed region
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        launches = _lib.launch_count() - launches0
        stages = None
        if with_stage_timer:
            _lib.timing_enable(False)
            stages = _lib.timing_read(reset=True)
        if world > 1:
            t = torch.tensor([ms], device=device, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, launches, stages, last

    sampler = ClockSampler(local) if rank == 0 else None
    ms_total, launches, stages, last = timed(step_resident, True)
    ms_eager = ms_total
    if args.cuda_graph:
        # the eager pass above supplies the per-stage events (they cannot be recorded inside a replay); the value is the replayed step
        for buf in dev_in:
            buf.copy_(raw)                                              # capture runs the step on the ring slots: give them real planes
        for cam in dev_cam:
            cam[0].copy_(c2w); cam[1].copy_(k)
        graphed = {"resident": graphs.capture(lambda: hot_path_step(torch, mods, raw, dec, c2w, k, res, opts)),
                   "slot": [graphs.capture(lambda s_=s_: hot_path_step(torch, mods, dev_in[s_], dec, dev_cam[s_][0], dev_cam[s_][1], res, opts))
                            for s_ in (0, 1)]}
        ms_total, _, _, last = timed(step_resident, False)
        launches = graphed["resident"].kernels * steps
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        # before the e2e steps: they reset the gradients and (N > 1) reuse the gathered buffers
        if train:
            dumped = {"loss": last, "grad_planes": raw.grad, **{f"grad_decoder.{n_}": p_.grad for n_, p_ in dec.named_parameters()}}
        else:
            maps = last.wait() if world > 1 else last
            dumped = {n_: t_ for n_, t_ in zip(("rgb", "seg", "depth", "wsum"), maps) if t_ is not None}
        dump_outputs(args.dump_outputs, dumped)
    del last
    ms_e2e, _, _, _ = timed(step_e2e, False)
    h2d_gbs = None if train else h2d_rate_concurrent()
    graph_extra = None
    if not args.cuda_graph and not train and world == 1 and rays_per_rank * (wl["s_c"] + wl["s_f"]) <= (1 << 26):
        # reported beside the eager numbers (never instead of them): the same resident step replayed as ONE CUDA graph
        from nerffaceediting_b200 import graphs
        try:        # an extra beside the contract's numbers (all measured above): it must never cost the line
            graphed = {"resident": graphs.capture(lambda: hot_path_step(torch, mods, raw, dec, c2w, k, res, opts)), "slot": None}
            ms_graph, _, _, _ = timed(step_resident, False)
            graph_extra = {"value": rays_per_rank / (ms_graph / steps * 1e-3), "unit": "rays/s", "ms_per_step": ms_graph / steps,
                           "kernels_per_replay": graphed["resident"].kernels,
                           "note": "same resident step captured once (nerffaceediting_b200.graphs.capture) and replayed with one launch per step; "
                                   "`value`, `e2e`, `roofline` and `stages_ms_per_step` above are the eager public-API calls"}
        except Exception as exc:    # noqa: BLE001
            graph_extra = {"error": f"{type(exc).__name__}: {exc}"[:300]}
        graphed = None

    # ---- extras beside the contract's numbers (single GPU, default workload only; each guarded: they must never cost the line)
    extras = {}
    if world == 1 and not train and not args.cuda_graph and args.workload == "c2" and not args.no_extras:
        def quick(fn, k_steps=10, k_warm=3):
            for _ in range(k_warm):
                fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(k_steps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / k_steps
        from nerffaceediting_b200 import ops as nfe_ops

        def torch_normalize(planes):
            mean = torch.mean(planes, dim=(-1, -2), keepdim=True)
            var = torch.sqrt(torch.var(planes, dim=(-1, -2), keepdim=True))
            return (planes - mean) / (var + 1e-8), mean, var
        try:
            # the TRUE drop-in flow of an unpickled generator (VERDICT r01 weak #3): its own torch normalize_plane
            # (training/triplane.py:56-65), our renderer without provenance -> both plane sets staged and gathered
            foreign = dict(mods, normalize_plane=torch_normalize)
            nfe_ops.path_counts(reset=True)
            with torch.no_grad():
                ms_f = quick(lambda: hot_path_step(torch, foreign, raw, dec, c2w, k, res, opts))
            extras["unpatched_generator"] = {"value": rays_per_rank / (ms_f * 1e-3), "unit": "rays/s", "ms_per_step": ms_f,
                                             "paths": nfe_ops.path_counts(reset=True),
                                             "note": "normalize_plane in plain torch ops (what an unpickled TriPlaneGenerator runs), renderer through "
                                                     "shadow/: no staging or provenance records, so planes_channel_last x2 + the two-gather field kernel"}
        except Exception as exc:    # noqa: BLE001
            extras["unpatched_generator"] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
        try:
            # the reference's own mode: stochastic stratified jitter + stochastic inverse-CDF draws (renderer.py:180-190,210-211)
            sto = dict(opts, nfe_deterministic=False)
            with torch.no_grad():
                ms_s = quick(lambda: hot_path_step(torch, mods, raw, dec, c2w, k, res, sto))
            extras["stochastic_sampling"] = {"value": rays_per_rank / (ms_s * 1e-3), "unit": "rays/s", "ms_per_step": ms_s,
                                             "note": "rendering_options without nfe_deterministic: in-kernel Philox jitter and u, as the reference always samples"}
        except Exception as exc:    # noqa: BLE001
            extras["stochastic_sampling"] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
        try:
            # BASELINE configs[3]: the training step (forward + backward), batch 32
            wl4 = WORKLOADS["c4"]
            raw4_host, dec4, c2w4, k4, opts4 = make_inputs(torch, wl4, torch.device("cpu"), 2000)
            opts4["nfe_precision"] = args.precision
            raw4 = raw4_host.to(device).requires_grad_(True)
            dec4 = dec4.to(device)
            c2w4, k4 = c2w4.to(device), k4.to(device)
            gw4 = torch.Generator(device="cpu").manual_seed(5)
            proj4 = [torch.randn(wl4["batch"], wl4["res"] ** 2, c, generator=gw4).to(device) for c in (32, 15, 1, 1)]

            def train4():
                raw4.grad = None
                for p_ in dec4.parameters():
                    p_.grad = None
                out = hot_path_step(torch, mods, raw4, dec4, c2w4, k4, wl4["res"], opts4)
                sum((o_ * w_).sum() for o_, w_ in zip(out, proj4)).backward()
            ms_4 = quick(train4, 5, 2)
            extras["c4_training_step"] = {"value": wl4["batch"] * wl4["res"] ** 2 / (ms_4 * 1e-3), "unit": "rays/s", "ms_per_step": ms_4,
                                          "workload": wl4["desc"]}
            del raw4, proj4
        except Exception as exc:    # noqa: BLE001
            extras["c4_training_step"] = {"error": f"{type(exc).__name__}: {exc}"[:300]}

        for name_x, k_x in (("c3", 5), ("c5", 3)):
            try:
                # the other BASELINE shapes, so that the driver's run times them too (VERDICT r01 weak #11): configs[2] (batch 32,
                # 128^2 rays) and configs[4] (one identity under 64 poses, 256^2 rays, 96+96 samples)
                wlx = WORKLOADS[name_x]
                rawx_host, decx, c2wx, kx_, optsx = make_inputs(torch, wlx, torch.device("cpu"), 3000)
                optsx["nfe_precision"] = args.precision
                rawx, decx, c2wx, kx_ = rawx_host.to(device), decx.to(device), c2wx.to(device), kx_.to(device)
                with torch.no_grad():
                    ms_x = quick(lambda: hot_path_step(torch, mods, rawx, decx, c2wx, kx_, wlx["res"], optsx), k_x, 2)
                rays_x = wlx["batch"] * wlx["res"] ** 2
                extras[name_x] = {"value": rays_x / (ms_x * 1e-3), "unit": "rays/s", "ms_per_step": ms_x, "workload": wlx["desc"],
                                  "samples_per_s": rays_x * (wlx["s_c"] + wlx["s_f"]) / (ms_x * 1e-3)}
                del rawx, rawx_host
                torch.cuda.empty_cache()
            except Exception as exc:    # noqa: BLE001
                extras[name_x] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
        try:
            # SURVEY.md §8f row f3: the consumer of the rendered feature image.  The default super-resolution head
            # (SuperresolutionHybrid8XDC, superresolution.py:264-290: 32 x 64^2 features -> 3 x 512^2, fp16 blocks as train.py sets
            # them) at this workload's batch, and its largest layer alone against the tensor roofline.
            import synth_inputs as synth
            from nerffaceediting_b200 import networks as nfe_net
            nb = wl["batch"]
            with torch.no_grad():
                sr = synth.fill_module(nfe_net.SuperresolutionHybrid8XDC(32, 512, 4, True), 3).to(device).eval()
                feat = torch.randn(nb, 32, res, res, device=device)
                ws_sr = torch.randn(nb, 14, 512, device=device)
                ms_sr = quick(lambda: sr(feat[:, :3].contiguous(), feat, ws_sr, noise_mode='const'), 5, 2)
                layer = synth.fill_module(nfe_net.SynthesisLayer(256, 256, w_dim=512, resolution=256, conv_clamp=256), 11).to(device).eval()
                xl = torch.randn(nb, 256, 256, 256, device=device, dtype=torch.float16).contiguous(memory_format=torch.channels_last)
                wl_ = torch.randn(nb, 512, device=device)
                ms_l = quick(lambda: layer(xl, wl_, noise_mode='const'), 10, 3)
            flop_l = 2.0 * nb * 256 * 256 * 9 * 256 * 256
            pk = measured_peaks()[2]
            tpeak = float(pk.get("bf16_tflops_sustained", 0) or 0)
            extras["f3_conv_stack"] = {
                "sr_head": {"value": nb / (ms_sr * 1e-3), "unit": "images/s", "ms": ms_sr, "workload": f"SuperresolutionHybrid8XDC, batch {nb}, fp16 blocks, 195.6 GFLOP of convolutions per image",
                            "conv_tflops": nb * 195.6 / ms_sr},
                "layer_256x256_at_256": {"ms": ms_l, "tflops": flop_l / ms_l / 1e9, "dtype": "f16 operands, f32 accumulate",
                                         "roofline": {"bound": "tensor", "achieved": flop_l / ms_l / 1e9, "peak": tpeak or None, "unit": "TFLOP/s",
                                                      "frac": (flop_l / ms_l / 1e9 / tpeak) if tpeak else None,
                                                      "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (dense 16-bit tensor rate)"}},
                "note": "modulated convolutions as tcgen05 implicit GEMMs (csrc/nfe_modconv.cu); the whole layer call is timed: weight fold + pack, "
                        "GEMM with fused noise / bias / lrelu / clamp epilogue"}
            del sr, feat, layer, xl
        except Exception as exc:    # noqa: BLE001
            extras["f3_conv_stack"] = {"error": f"{type(exc).__name__}: {exc}"[:300]}

        for tag_g, g16 in (("full_generator", 0), ("full_generator_fp16_backbone", 4)):
            try:
                # BASELINE configs[1] in full: mapping + StyleGAN2 tri-plane backbone + decoders + renderer + super-resolution, 512^2 output,
                # 64^2 neural resolution, batch 8 — this package's TriPlaneGenerator with the reference's default sizes (train.py:150-151,
                # 183-184,225-245,343-355: cbase 32768, cmax 512, map depth 2, fp32 backbone, fp16 super-resolution blocks).  The second
                # variant runs the backbone's high resolutions in fp16 as well (--g_num_fp16_res 4).
                import synth_inputs as synth
                from nerffaceediting_b200 import triplane as nfe_triplane
                rk = dict(synth.FFHQ_RENDERING_OPTIONS, superresolution_module='training.superresolution.SuperresolutionHybrid8XDC', sr_antialias=True,
                          superresolution_noise_mode='none', c_gen_conditioning_zero=False, c_scale=1.0, decoder_lr_mul=1, nfe_deterministic=True,
                          nfe_precision=args.precision)
                nb = wl["batch"]
                with torch.no_grad():
                    G = nfe_triplane.TriPlaneGenerator(z_dim=512, c_dim=25, w_dim=512, img_resolution=512, img_channels=3, sr_num_fp16_res=4,
                                                       mapping_kwargs=dict(num_layers=2), rendering_kwargs=rk, channel_base=32768, channel_max=512,
                                                       num_fp16_res=g16, conv_clamp=256 if g16 else None, fused_modconv_default='inference_only',
                                                       sr_kwargs=dict(channel_base=32768, channel_max=512, fused_modconv_default='inference_only'))
                    G = synth.fill_module(G, 77).to(device).eval()
                    zg = torch.randn(nb, 512, device=device)
                    cam = torch.cat([c2w.reshape(nb, 16), k.reshape(nb, 9)], dim=1).float()
                    ms_g = quick(lambda: G(zg, cam, noise_mode='const'), 5, 2)
                    # the same through host buffers: latents and cameras up from pinned memory, the images (and the raw / semantic /
                    # depth maps) back into pinned memory, every step
                    z_host, cam_host = zg.cpu().pin_memory(), cam.cpu().pin_memory()
                    outs_host = {}

                    def g_e2e():
                        zd, cd = z_host.to(device, non_blocking=True), cam_host.to(device, non_blocking=True)
                        o_ = G(zd, cd, noise_mode='const')
                        for kk_ in ('image', 'image_seg', 'image_raw', 'image_depth'):
                            if kk_ not in outs_host:
                                outs_host[kk_] = torch.empty(o_[kk_].shape, dtype=o_[kk_].dtype).pin_memory()
                            outs_host[kk_].copy_(o_[kk_], non_blocking=True)
                    ms_ge = quick(g_e2e, 5, 2)
                    d2h_g = sum(v.numel() * v.element_size() for v in outs_host.values())
                extras[tag_g] = {"value": rays_per_rank / (ms_g * 1e-3), "unit": "rays/s", "images_per_s": nb / (ms_g * 1e-3), "ms_per_step": ms_g,
                                 "e2e": {"value": rays_per_rank / (ms_ge * 1e-3), "unit": "rays/s", "images_per_s": nb / (ms_ge * 1e-3), "ms_per_step": ms_ge,
                                         "h2d_bytes_per_step": int(z_host.numel() * 4 + cam_host.numel() * 4), "d2h_bytes_per_step": int(d2h_g)},
                                 "workload": f"configs[1] full generator synthesis: batch {nb}, 512^2 output, 64^2 neural resolution, 48+48 samples, "
                                             f"backbone {'fp16 from 32^2 up' if g16 else 'fp32 (bf16x3 tensor-core arithmetic)'}, super-resolution fp16, "
                                             "random-init weights"}
                del G
                torch.cuda.empty_cache()
            except Exception as exc:    # noqa: BLE001
                extras[tag_g] = {"error": f"{type(exc).__name__}: {exc}"[:300]}

    if rank == 0:
        ms_step = ms_total / steps
        total_rays = rays_per_rank * world
        value = total_rays / (ms_step * 1e-3)
        e2e_value = total_rays / (ms_e2e / steps * 1e-3)
        # dominant kernel: the fused gather+decode field kernel (coarse + fine launches)
        f_ms = stages["field_coarse"][0] + stages["field_fine"][0]
        f_n = stages["field_coarse"][1] + stages["field_fine"][1]
        # the host splits a call whose workspace would exceed NFE_WORKSPACE_MB into item chunks (c3, c5): count the launches that
        # actually ran, every sample of the timed steps being gathered + decoded exactly once
        samples_per_launch = rays_per_rank * (wl["s_c"] + wl["s_f"]) * steps / max(f_n, 1)
        alg_bytes = samples_per_launch * sets_gathered * GATHER_BYTES_PER_SAMPLE_SET
        avg_ms = f_ms / max(f_n, 1)
        achieved = alg_bytes / (avg_ms * 1e-3) / 1e9
        peak, peak_src, peaks = measured_peaks()
        traffic = None
        tp = os.path.join(ROOT, "profiles", "field_kernel_traffic.json")
        if os.path.exists(tp):
            try:
                traffic = json.load(open(tp)).get("dram_bytes_per_launch")
            except Exception:
                traffic = None
        # ---- governing roofline of the field kernel (SURVEY.md §8d): t_min = max(compulsory HBM bytes / BW_HBM,
        #      gather bytes / BW_L2, MLP flops issued / tensor peak); BW_L2 is measured live (measure_l2_gather)
        try:
            l2 = measure_l2_gather(torch, _lib, device)
        except Exception as exc:    # noqa: BLE001
            l2 = {"error": f"{type(exc).__name__}: {exc}"[:200]}
        l2_peak = l2.get("peak")
        pb = wl.get("plane_batch", n)
        launches_per_step = max(f_n, 1) / steps
        set_bytes = 3 * 32 * 256 * 256 * 4
        # the plane sets a launch reads, once each (a call split into item chunks reads its own items; a shared set is read by every launch)
        plane_bytes = sets_gathered * set_bytes * (1 if pb == 1 else pb / max(launches_per_step / 2, 1))
        compulsory = plane_bytes + samples_per_launch * (4 + 192 + 4) + samples_per_launch / wl["s_c"] * 24  # + depths in, records + sigma out, rays
        mma_mult = {"bf16x3": 3.0, "bf16": 1.0}.get(args.precision)
        flops = samples_per_launch * MLP_FLOP_PER_SAMPLE
        tensor_peak = float(peaks.get("bf16_tflops_sustained") or peaks.get("bf16_tflops") or 0.0)
        terms = {"hbm": compulsory / (peak * 1e9) * 1e3}
        if l2_peak:
            terms["l2"] = alg_bytes / (l2_peak * 1e9) * 1e3
        if mma_mult and tensor_peak > 0:
            terms["tensor"] = flops * mma_mult / (tensor_peak * 1e12) * 1e3
        bound = max(terms, key=terms.get)
        t_min = terms[bound]
        if bound == "tensor":
            roof_achieved, roof_peak, roof_unit = flops * mma_mult / (avg_ms * 1e-3) / 1e12, tensor_peak, "TFLOP/s"
        elif bound == "l2":
            roof_achieved, roof_peak, roof_unit = achieved, l2_peak, "GB/s"
        else:
            roof_achieved, roof_peak, roof_unit = compulsory / (avg_ms * 1e-3) / 1e9, peak, "GB/s"
        line = {
            "metric": f"rendered rays/sec ({wl['s_c']}+{wl['s_f']} samples)" + (", forward+backward" if train else ""), "value": value, "unit": "rays/s", "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": dtype, "data": "synthetic",
            "config": {"workload": wl["desc"], "rays_per_gpu_per_step": rays_per_rank, "sampling": "deterministic (parity mode)",
                       "sample": "the whole workload every step",
                       "parallelism": (f"batch-sharded x{world} through nerffaceediting_b200.sharding.ShardedRenderer: NCCL all-gather of the rendered maps "
                                       "overlapped on a communication stream") if world > 1 else "single GPU",
                       "cache": ("one 25 MB plane set stays L2-resident by design (one identity, many poses); the per-step stream of per-sample records "
                                 "(chunked workspace, GBs) and the 822 MB of output maps pass through L2 between steps, no separate flush") if wl.get("plane_batch") == 1 else
                                "inputs larger than L2 (raw+normalised+staged planes ~0.8 GB per step), no L2 flush needed"},
            "e2e": {"value": e2e_value, "unit": "rays/s", "ms_per_step": ms_e2e / steps,
                    "h2d_bytes_per_step": int(raw_host.numel() * 4 + c2w_host.numel() * 4 + k_host.numel() * 4),
                    "d2h_bytes_per_step": 4 if train else int(out_host[0].numel() * 4),
                    "h2d_gbs_per_rank_all_ranks_uploading": h2d_gbs, "numa": numa,
                    "note": "training step: planes + cameras uploaded, loss scalar read back, every step" if train else
                            "uploads double-buffered (step i+1's H2D overlaps step i's render), in batch-item chunks over two copy streams; "
                            "bound by the host->device link: h2d_gbs_per_rank_all_ranks_uploading is the rate the slowest rank gets while all "
                            "ranks upload at once, i.e. the ceiling of e2e = h2d_bytes_per_step / that rate"},
            "gpu_launches": launches,
            "roofline": {"kernel": "field_pipe2_kernel<disentangled> (tri-plane gather + decoder MLPs), coarse+fine launches", "bound": bound,
                         "achieved": roof_achieved, "peak": roof_peak, "unit": roof_unit, "frac": t_min / avg_ms, "traffic": traffic,
                         "t_min_ms": t_min, "t_min_terms_ms": terms, "avg_launch_ms": avg_ms,
                         "peak_source": ("nfe_bench_l2_gather, measured in this run: random 128-byte lines of an L2-resident 25 MB table, LDG.128, "
                                         "32 warps x 8 loads in flight per SM" if bound == "l2" else peak_src),
                         "l2_gbs_measured": l2,
                         "algorithmic_bytes_per_launch": alg_bytes, "compulsory_hbm_bytes_per_launch": compulsory,
                         "hbm": {"achieved": achieved, "peak": peak, "frac": achieved / peak, "peak_source": peak_src,
                                 "note": "algorithmic gather bytes / kernel time against the measured HBM copy peak (round 1's figure; the gather "
                                         "is served by L2, so this can exceed 1 and is not the governing roof)"},
                         "mlp_tflops": flops / (avg_ms * 1e-3) / 1e12,
                         "mlp_tensor_frac": tensor_frac(flops / (avg_ms * 1e-3) / 1e12, args.precision, peaks),
                         "share_of_step": f_ms / ms_eager,
                         "plane_sets_gathered": sets_gathered,
                         "note": "frac = t_min / measured launch time with t_min = max(compulsory HBM bytes / measured HBM peak, gather bytes / "
                                 "measured L2 gather bandwidth, MMA flops issued / sustained bf16 peak); gather bytes = 1536 B per sample per "
                                 "plane set actually gathered (the single-gather identity reads one set; the reference's formulation reads two)"},
            "stages_ms_per_step": {k_: v[0] / steps for k_, v in stages.items() if v[1]},
            "clocks": clocks,
        }
        if args.swap_statistics:
            line["config"]["statistics_swap"] = "denormalize_plane(norm, roll(mean), roll(std)) inside the step"
        if graph_extra is not None:
            line["cuda_graph"] = graph_extra
        if extras:
            line["extras"] = extras
        if args.cuda_graph:
            line["cuda_graph"] = {"kernels_per_replay": graphed["resident"].kernels, "eager_ms_per_step": ms_eager / steps,
                                  "note": "value and e2e replay the step as one CUDA graph; roofline and stages come from the eager pass of the "
                                          "same steps run just before (stage events cannot be recorded inside a replay)"}
            line["config"]["cuda_graph"] = True
        if world == 1 and not args.no_cpu_baseline and not train:   # the CPU port is forward-only
            r = cpu_reference_rate(torch, wl, 3, 1)
            line["cpu_baseline"] = {"value": r["rays_per_s_best"], "unit": "rays/s", "cores": r["cores"], "kind": "port", "sample": r["sample"] + " (best)"}
            if wl["res"] <= 64:                                        # the scalar figure SURVEY.md §8d also asks for (one more bounded step)
                r1 = cpu_reference_rate(torch, wl, 1, 0, threads=1)
                line["cpu_baseline"]["one_thread_value"] = r1["rays_per_s_best"]
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
