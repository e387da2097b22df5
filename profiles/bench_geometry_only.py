"""Full against geometry-only renders (rendering_options['nfe_geometry_only']) on the bench workloads c2, c3 and c5 with the
DisentangledOSGDecoder, and c2 with the SegmentationOSGDecoder (reported as `c2_seg`).

    python profiles/bench_geometry_only.py [--steps-c2 20] [--steps-c3 5] [--steps-c5 2] [--reps 3] [--out result.json]

For every disentangled workload two plane flows are measured: 'package' (normalize_plane of this package: the full render takes the
single-gather identity) and 'foreign' (normalised in plain torch ops, what an unpatched generator runs: the full render stages and
gathers both plane sets).  The segmentation decoder reads the raw planes alone, so it runs the 'package' flow only.  Full and
geometry-only steps (RaySampler -> normalize_plane -> renderer, bench.py's hot-path call) are alternated in one process, `reps` rounds of `steps` timed steps each after a warm-up; the reported step time is the median round,
the per-stage times come from the library's stage timer (nfe_timing_*) over the same steps.  seg / depth / wsum of the last steps
are checked to be bit-identical between the two modes.  The JSON carries the GPU name and power limit read in the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def gpu_identity(torch):
    info = {"name": torch.cuda.get_device_name(0), "power_limit_w": None, "sm_clock_max_mhz": None}
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        info["power_limit_w"], info["sm_clock_max_mhz"] = float(out[0]), float(out[1])
    except (OSError, ValueError, IndexError, subprocess.SubprocessError) as exc:
        info["error"] = f"{type(exc).__name__}: {exc}"[:160]
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps-c2", type=int, default=20)
    ap.add_argument("--steps-c3", type=int, default=5)
    ap.add_argument("--steps-c5", type=int, default=2)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from bench import WORKLOADS, hot_path_step, make_inputs
    from nerffaceediting_b200 import _lib, triplane
    from nerffaceediting_b200.ray_sampler import RaySampler
    from nerffaceediting_b200.renderer import DisentangledImportanceRenderer
    from nerffaceediting_b200.triplane import SegmentationOSGDecoder
    if not torch.cuda.is_available():
        raise SystemExit("bench_geometry_only: needs a CUDA device")
    device = torch.device("cuda:0")

    def torch_normalize(planes):
        mean = torch.mean(planes, dim=(-1, -2), keepdim=True)
        std = torch.sqrt(torch.var(planes, dim=(-1, -2), keepdim=True))
        return (planes - mean) / (std + 1e-8), mean, std

    result = {"gpu": gpu_identity(torch), "reps": args.reps, "workloads": {}}
    for name, wl_name, decoder in (("c2", "c2", "dis"), ("c2_seg", "c2", "seg"), ("c3", "c3", "dis"), ("c5", "c5", "dis")):
        wl = WORKLOADS[wl_name]
        steps = {"c2": args.steps_c2, "c3": args.steps_c3, "c5": args.steps_c5}[wl_name]
        raw_host, dec, c2w, k, opts = make_inputs(torch, wl, device, 1000)
        if decoder == "seg":
            torch.manual_seed(1000)
            dec = SegmentationOSGDecoder(32, {'decoder_lr_mul': 1, 'decoder_output_dim': 32, 'decoder_seg_dim': 15})
        raw, dec, c2w, k = raw_host.to(device), dec.to(device), c2w.to(device), k.to(device)
        rays = wl["batch"] * wl["res"] ** 2
        base = {"sampler": RaySampler(), "renderer": DisentangledImportanceRenderer()}
        flows = {"package": dict(base, normalize_plane=triplane.normalize_plane), "foreign": dict(base, normalize_plane=torch_normalize)}
        if decoder == "seg":
            del flows["foreign"]
        modes = {"full": opts, "geometry_only": dict(opts, nfe_geometry_only=True)}
        times = {(f, m): [] for f in flows for m in modes}
        stage_ms = {(f, m): {} for f in flows for m in modes}
        last = {}
        with torch.no_grad():
            for f, mods in flows.items():                               # warm-up: first launches, allocator growth
                for m, o in modes.items():
                    last[(f, m)] = hot_path_step(torch, mods, raw, dec, c2w, k, wl["res"], o)
            torch.cuda.synchronize()
            for _ in range(args.reps):
                for f, mods in flows.items():
                    for m, o in modes.items():
                        del last[(f, m)]
                        _lib.timing_read(reset=True)
                        _lib.timing_enable(True)
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        e0.record()
                        for _ in range(steps):
                            out = hot_path_step(torch, mods, raw, dec, c2w, k, wl["res"], o)
                        e1.record()
                        torch.cuda.synchronize()
                        _lib.timing_enable(False)
                        times[(f, m)].append(e0.elapsed_time(e1) / steps)
                        for st, (ms, cnt) in _lib.timing_read(reset=True).items():
                            if cnt:
                                stage_ms[(f, m)].setdefault(st, []).append(ms / steps)
                        last[(f, m)] = out
        for f in flows:
            full, geo = last[(f, "full")], last[(f, "geometry_only")]
            assert geo[0] is None and all(torch.equal(a, b) for a, b in zip(full[1:], geo[1:])), (name, f)
        entry = {"desc": wl["desc"] + ("" if decoder == "dis" else "; SegmentationOSGDecoder instead"), "rays_per_step": rays,
                 "steps_per_round": steps, "flows": {}}
        for f in flows:
            entry["flows"][f] = {}
            for m in modes:
                ms = statistics.median(times[(f, m)])
                entry["flows"][f][m] = {"ms_per_step": ms, "ms_per_step_rounds": times[(f, m)], "rays_per_s": rays / (ms * 1e-3),
                                        "stages_ms_per_step": {st: statistics.median(v) for st, v in stage_ms[(f, m)].items()}}
            entry["flows"][f]["step_speedup"] = entry["flows"][f]["full"]["ms_per_step"] / entry["flows"][f]["geometry_only"]["ms_per_step"]
        result["workloads"][name] = entry
        print(json.dumps({name: {f: {m: round(v["ms_per_step"], 3) for m, v in e.items() if isinstance(v, dict)}
                                 for f, e in entry["flows"].items()}}), flush=True)
        del raw, last
        torch.cuda.empty_cache()
    text = json.dumps(result, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
