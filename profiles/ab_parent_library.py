"""Default-path step times of this tree's libnfe_b200.so against another build of it (e.g. the parent commit's), alternated in one
process, with the outputs of the two compared bit for bit.

    # build the other revision in a separate checkout: python -m nerffaceediting_b200.build, then
    python profiles/ab_parent_library.py --other /path/to/other/nerffaceediting_b200/lib/libnfe_b200.so [--out result.json]

Both libraries are loaded with this tree's ctypes prototypes and the Python layer switches between them step by step (the
nfe_render_cfg struct only grows at its end, so an older library reads the fields it knows).  Workloads c2 (20 steps) and c3
(5 steps) of bench.py, full renders in the package flow, 6 rounds with the order of the two libraries alternated.  The JSON
carries the GPU name and power limit read in the same run.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--other", required=True, help="the other build's libnfe_b200.so")
    ap.add_argument("--label", default=None, help="what the other build is (stored in the JSON; default: the path)")
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from bench import WORKLOADS, hot_path_step, make_inputs
    from nerffaceediting_b200 import _lib, triplane
    from nerffaceediting_b200.ray_sampler import RaySampler
    from nerffaceediting_b200.renderer import DisentangledImportanceRenderer
    if not torch.cuda.is_available():
        raise SystemExit("ab_parent_library: needs a CUDA device")
    libs = {}
    for tag, path in (("other", args.other), ("this", _lib.LIB_PATH)):
        lib = ctypes.CDLL(os.path.abspath(path))
        for name, (res, argtypes) in _lib.SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, argtypes
        libs[tag] = lib
    dev = torch.device("cuda:0")
    gpu = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip()
    out = {"gpu": gpu, "other": args.label or args.other, "workloads": {}}
    try:
        for name, steps in (("c2", 20), ("c3", 5)):
            wl = WORKLOADS[name]
            raw_h, dec, c2w, k, opts = make_inputs(torch, wl, dev, 1000)
            raw, dec, c2w, k = raw_h.to(dev), dec.to(dev), c2w.to(dev), k.to(dev)
            mods = {"sampler": RaySampler(), "renderer": DisentangledImportanceRenderer(), "normalize_plane": triplane.normalize_plane}
            times, last = {"other": [], "this": []}, {}
            with torch.no_grad():
                for tag in libs:                                   # warm-up of both
                    _lib._lib = libs[tag]
                    for _ in range(3):
                        last[tag] = hot_path_step(torch, mods, raw, dec, c2w, k, wl["res"], opts)
                torch.cuda.synchronize()
                for rnd in range(args.rounds):
                    for tag in (("other", "this") if rnd % 2 == 0 else ("this", "other")):
                        _lib._lib = libs[tag]
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        e0.record()
                        for _ in range(steps):
                            o = hot_path_step(torch, mods, raw, dec, c2w, k, wl["res"], opts)
                        e1.record()
                        torch.cuda.synchronize()
                        times[tag].append(e0.elapsed_time(e1) / steps)
                        last[tag] = o
            same = all(torch.equal(a, b) for a, b in zip(last["other"], last["this"]))
            out["workloads"][name] = {"ms_per_step_median": {t: statistics.median(v) for t, v in times.items()}, "rounds": times,
                                      "outputs_equal": same}
            print(name, json.dumps(out["workloads"][name]), flush=True)
            del raw, last
    finally:
        _lib._lib = libs["this"]
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
