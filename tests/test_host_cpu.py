"""CPU-side tests: the C-ABI library loads and exports what include/nfe_b200.h declares, the host
logic (decoder recognition, option handling, shadow package) behaves, and nothing falls back to a CPU
compute path.  No kernel is launched here."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from nerffaceediting_b200 import _lib, ops
import synth_inputs as synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# a checkout of the original NeRFFaceEditing project; the tests that import its modules skip without one
REFERENCE = os.environ.get("NFE_REFERENCE", "")
needs_reference = pytest.mark.skipif(not (REFERENCE and os.path.isdir(os.path.join(REFERENCE, "training"))),
                                     reason="needs a checkout of the original NeRFFaceEditing project in $NFE_REFERENCE")


@pytest.fixture(scope="module")
def built():
    from nerffaceediting_b200 import build
    return build.build()


def header_functions():
    text = open(os.path.join(ROOT, "include", "nfe_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(nfe_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol(built):
    names = header_functions()
    assert len(names) >= 20
    lib = ctypes.CDLL(built)
    for name in names:
        assert hasattr(lib, name), f"{name} declared in include/nfe_b200.h but not exported"
        assert name in _lib.SIGNATURES, f"{name} has no ctypes prototype in _lib.SIGNATURES"
    assert sorted(_lib.SIGNATURES) == names
    assert _lib.load().nfe_version() == 1
    assert isinstance(_lib.launch_count(), int)


def test_library_is_sm100a_only(built):
    out = subprocess.run(["cuobjdump", "-lelf", built], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, archs


def test_struct_layouts_match_header():
    # nfe_mlp: 4 pointers, 3 ints, 4 floats; nfe_render_cfg ends with precision after two uint64
    assert ctypes.sizeof(_lib.NfeMlp) == 4 * 8 + 3 * 4 + 4 * 4 + 4   # trailing pad to 8
    assert _lib.NfeRenderCfg.seed.offset % 8 == 0 and _lib.NfeRenderCfg.precision.offset == _lib.NfeRenderCfg.offset.offset + 8


def test_no_cpu_fallback():
    from nerffaceediting_b200 import triplane
    from nerffaceediting_b200.ray_sampler import RaySampler
    from nerffaceediting_b200.renderer import ImportanceRenderer, sample_from_planes
    with pytest.raises(RuntimeError, match="CUDA"):
        triplane.normalize_plane(torch.randn(1, 96, 8, 8))
    with pytest.raises(RuntimeError, match="CUDA"):
        RaySampler()(torch.eye(4)[None], torch.eye(3)[None], 4)
    with pytest.raises(RuntimeError, match="CUDA"):
        sample_from_planes(None, torch.randn(1, 3, 32, 8, 8), torch.zeros(1, 2, 3), box_warp=1)
    dec = triplane.OSGDecoder(32, {'decoder_lr_mul': 1, 'decoder_output_dim': 32})
    with pytest.raises(RuntimeError, match="CUDA"), torch.no_grad():
        ImportanceRenderer()(torch.randn(1, 3, 32, 8, 8), dec, torch.zeros(1, 2, 3), torch.ones(1, 2, 3), synth.FFHQ_RENDERING_OPTIONS)


def test_graph_capture_needs_cuda():
    from nerffaceediting_b200 import graphs
    if torch.cuda.is_available():
        pytest.skip("CPU-container check")
    with pytest.raises(RuntimeError, match="CUDA"):
        graphs.capture(lambda: None)


def test_bench_workloads_cover_every_baseline_config():
    """bench.py names one workload per BASELINE.json config (c1..c5) and the reference arm runs the oracle port on them."""
    import json
    import bench
    configs = json.load(open(os.path.join(ROOT, "BASELINE.json")))["configs"]
    assert sorted(bench.WORKLOADS) == [f"c{i + 1}" for i in range(len(configs))]
    assert bench.WORKLOADS["c5"]["plane_batch"] == 1 and bench.WORKLOADS["c5"]["res"] == 256 and bench.WORKLOADS["c5"]["s_c"] == 96
    raw, dec, c2w, k, opts = bench.make_inputs(torch, dict(bench.WORKLOADS["c5"], batch=2), torch.device("cpu"), 0)
    assert raw.shape == (1, 96, 256, 256) and c2w.shape == (2, 4, 4) and opts["depth_resolution_importance"] == 96


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside ours): ONE JSON line on stdout with the contract's keys,
    timed on the oracle port with the host's threads, no GPU needed."""
    import json
    import subprocess
    import sys
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "rays/s" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["metric"] == "rendered rays/sec (48+48 samples)" and d["value"] > 0 and d["gpu_launches"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # ranks other than 0 of a torchrun launch exit without work or output
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, env=dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1", CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_plane_registries_key_on_version_and_tolerate_inference_tensors():
    """The staging / provenance registries key on (address, shape, version): a 4-D tensor and its 5-D view share a key, an
    in-place write invalidates it, and tensors made under torch.inference_mode() (no version counter) simply never hit."""
    from nerffaceediting_b200 import ops
    from nerffaceediting_b200 import plane_registry as reg
    reg.clear()
    norm, raw = torch.randn(2, 96, 4, 4), torch.randn(2, 96, 4, 4)
    assert reg.key5(norm) == reg.key5(norm.view(2, 3, 32, 4, 4))
    reg.provenance_put(raw, norm, torch.ones(2, 96), torch.zeros(2, 96))
    hit = ops.provenance(norm.view(2, 3, 32, 4, 4), raw.view(2, 3, 32, 4, 4))
    assert hit is not None and hit[0].shape == (2, 96)
    assert ops.provenance(raw, norm) is None                     # the pair is ordered
    raw.add_(1.0)                                               # stale: the version moved on
    assert ops.provenance(norm, raw) is None
    with torch.inference_mode():
        n2, r2 = torch.randn(1, 96, 4, 4), torch.randn(1, 96, 4, 4)
        before = len(reg.PROVENANCE)
        reg.provenance_put(r2, n2, torch.ones(1, 96), torch.zeros(1, 96))
        assert len(reg.PROVENANCE) == before and ops.provenance(n2, r2) is None
        reg.staged_put(n2, n2)
        assert reg.staged_get(n2) is None
    reg.clear()


def test_plane_registries_never_hit_a_recycled_address():
    """ADVICE r01: an entry must die with the tensors it describes.  Tensors that land on a freed tensor's address (the
    caching allocator recycles blocks; here the same storage is re-wrapped) do not inherit its provenance or staging."""
    import gc
    from nerffaceediting_b200 import ops
    from nerffaceediting_b200 import plane_registry as reg
    reg.clear()
    pool_n, pool_r = torch.zeros(2 * 96 * 16), torch.zeros(2 * 96 * 16)      # stand-ins for allocator blocks
    norm, raw = pool_n.view(2, 96, 4, 4), pool_r.view(2, 96, 4, 4)
    reg.provenance_put(raw, norm, torch.full((2, 96), 2.0), torch.zeros(2, 96))
    reg.staged_put(norm, torch.ones(1))
    assert ops.provenance(norm, raw) is not None and reg.staged_get(norm) is not None
    key_n, key_r = reg.key5(norm), reg.key5(raw)
    del norm, raw
    gc.collect()
    norm_other, raw_other = pool_n.view(2, 96, 4, 4), pool_r.view(2, 96, 4, 4)   # same address, shape, version: other tensors
    assert reg.key5(norm_other) == key_n and reg.key5(raw_other) == key_r
    assert ops.provenance(norm_other, raw_other) is None
    assert reg.staged_get(norm_other) is None
    assert len(reg.PROVENANCE) == 0 and len(reg.STAGED) == 0                    # dead entries are dropped on lookup
    # ... while views and the registered objects themselves keep hitting
    norm, raw = torch.randn(2, 96, 4, 4), torch.randn(2, 96, 4, 4)
    reg.provenance_put(raw, norm, torch.ones(2, 96), torch.zeros(2, 96))
    v_n, v_r = norm.view(2, 3, 32, 4, 4), raw.view(2, 3, 32, 4, 4)
    del norm, raw
    gc.collect()
    assert ops.provenance(v_n, v_r) is not None                                 # a view keeps its base alive
    ops.clear_plane_cache()
    assert ops.provenance(v_n, v_r) is None and len(reg.SOURCES) == 0


def test_plane_registries_capacity_epochs_and_counters():
    """Several generators (G, G_ema, swap variants) coexist up to MAX_ENTRIES; a new epoch (graphs.capture) hides entries made
    before it and retires those made inside it; counts() reports which path calls took."""
    from nerffaceediting_b200 import plane_registry as reg
    reg.clear()
    reg.counts(reset=True)
    pairs = [(torch.randn(1, 96, 2, 2), torch.randn(1, 96, 2, 2)) for _ in range(reg.MAX_ENTRIES + 2)]
    for n_, r_ in pairs:
        reg.provenance_put(r_, n_, torch.ones(1, 96), torch.zeros(1, 96))
    assert len(reg.PROVENANCE) == reg.MAX_ENTRIES
    assert reg.provenance(*pairs[0]) is None and reg.provenance(*pairs[1]) is None       # the oldest two left
    assert all(reg.provenance(n_, r_) is not None for n_, r_ in pairs[2:])               # alternating between the rest never thrashes
    n0, r0 = pairs[-1]
    with reg.new_epoch():
        assert reg.provenance(n0, r0) is None                      # made before the capture: invisible inside
        n1, r1 = torch.randn(1, 96, 2, 2), torch.randn(1, 96, 2, 2)
        reg.provenance_put(r1, n1, torch.ones(1, 96), torch.zeros(1, 96))
        assert reg.provenance(n1, r1) is not None                  # made inside: visible inside
    assert reg.provenance(n1, r1) is None                          # ... and retired with the capture
    reg.note("render", "single-gather")
    reg.note("render", "single-gather")
    reg.note("render", "two-gather")
    c = reg.counts(reset=True)
    assert c["render:single-gather"] == 2 and c["render:two-gather"] == 1 and reg.counts() == {}
    reg.clear()


def test_plane_registries_resolve_batch_slices():
    """sharding / chunking pass batch slices of the generator's planes: they inherit staging and provenance, sliced alike."""
    from nerffaceediting_b200 import plane_registry as reg
    reg.clear()
    norm, raw = torch.randn(4, 96, 2, 2), torch.randn(4, 96, 2, 2)
    scale, shift = torch.arange(4 * 96.0).reshape(4, 96), -torch.arange(4 * 96.0).reshape(4, 96)
    reg.provenance_put(raw, norm, scale, shift)
    reg.staged_put(norm, torch.arange(4.0).reshape(4, 1).expand(4, 5).contiguous())
    n5, r5 = norm.view(4, 3, 32, 2, 2), raw.view(4, 3, 32, 2, 2)
    hit = reg.provenance(n5[1:3], r5[1:3])
    assert hit is not None and torch.equal(hit[0], scale[1:3]) and torch.equal(hit[1], shift[1:3])
    assert reg.provenance(n5[1:3], r5[2:4]) is None            # different slices of the pair
    assert reg.provenance(n5[0:2], r5[0:2]) is not None
    st = reg.staged_get(n5[2:4])
    assert st is not None and torch.equal(st[:, 0], torch.tensor([2.0, 3.0]))
    assert reg.staged_get(n5[:, 1:2]) is None                  # not a batch slice
    # one statistics row for the whole batch (triplane.py:100-101): every slice shares it
    out = torch.randn(4, 96, 2, 2)
    reg.provenance_put(out, norm, scale[:1], shift[:1])
    hit = reg.provenance(n5[3:4], out.view(4, 3, 32, 2, 2)[3:4])
    assert hit is not None and hit[0].shape == (1, 96)
    raw.add_(1)                                                 # an in-place write to the root invalidates its slices too
    assert reg.provenance(n5[1:3], r5[1:3]) is None
    reg.clear()


def test_plane_registries_are_thread_safe():
    import threading
    from nerffaceediting_b200 import plane_registry as reg
    reg.clear()
    errors = []

    def worker(seed):
        try:
            g = torch.Generator().manual_seed(seed)
            for _ in range(200):
                n_, r_ = torch.randn(1, 96, 2, 2, generator=g), torch.randn(1, 96, 2, 2, generator=g)
                reg.provenance_put(r_, n_, torch.ones(1, 96), torch.zeros(1, 96))
                hit = reg.provenance(n_, r_)
                assert hit is None or hit[0].shape == (1, 96)
                reg.staged_put(n_, r_)
                reg.staged_get(n_)
        except Exception as e:      # noqa: BLE001
            errors.append(e)
    threads = [threading.Thread(target=worker, args=(i,)) for i in range(4)]
    [t.start() for t in threads]
    [t.join() for t in threads]
    assert not errors
    reg.clear()


def test_field_plan_decision_table(monkeypatch):
    """renderer.field_plan over its table: when the single-gather identity applies, geometry-only, which plane sets are
    staged and which path counter a call records."""
    from nerffaceediting_b200 import plane_registry as reg
    from nerffaceediting_b200.renderer import field_plan
    reg.clear()
    monkeypatch.delenv("NFE_BWD_LIBRARY_GEMM", raising=False)
    monkeypatch.delenv("NFE_DEFAULT_PRECISION", raising=False)
    dis, osg = (ops.DEC_DISENTANGLED, None, None), (ops.DEC_OSG, None, None)
    norm, raw = torch.randn(2, 96, 4, 4), torch.randn(2, 96, 4, 4)
    reg.provenance_put(raw, norm, torch.full((2, 96), 2.0), torch.ones(2, 96))
    n5, r5, other = norm.view(2, 3, 32, 4, 4), raw.view(2, 3, 32, 4, 4), torch.randn(2, 3, 32, 4, 4)
    opts = dict(depth_resolution=48, depth_resolution_importance=48)

    def plan(what, desc, pair, per_item, grad=False, sigma_only=False, **o):
        p = field_plan(what, desc, *pair, dict(opts, **o), 2, per_item, grad, sigma_only)
        return p.affine is not None, p.geo_only, (p.stage_norm, p.stage_denorm), p.path

    single, two = (True, False, (True, False), ("render", "single-gather")), (False, False, (True, True), ("render", "two-gather"))
    assert plan("render", dis, (n5, r5), 64) == single
    assert plan("render", dis, (n5, r5), 64, nfe_precision="bf16") == single
    assert plan("render", dis, (n5, r5), 64, nfe_precision="fp32") == two               # fp32 never uses the identity
    assert plan("render", dis, (n5, r5), 64, nfe_single_gather=False) == two
    assert plan("render", dis, (n5, other), 64) == two                                  # no provenance
    assert plan("render", osg, (None, r5), 64) == (False, False, (False, True), ("render", "one-set"))
    # 128 samples per item in each pass: rays x min(coarse, fine) for a render, points for run_model
    assert plan("render", dis, (n5, r5), 3) == single                                   # 3 x 48
    assert plan("render", dis, (n5, r5), 3, depth_resolution_importance=40) == two      # 3 x 40
    assert plan("render", dis, (n5, r5), 3, depth_resolution=40) == two                 # 3 x 40
    assert plan("render", dis, (n5, r5), 2, depth_resolution_importance=0) == two       # 2 x 48, one pass
    assert plan("render", dis, (n5, r5), 1, depth_resolution=128, depth_resolution_importance=0) == single
    assert plan("render", dis, (n5, r5), 1, depth_resolution=127, depth_resolution_importance=0) == two
    assert plan("run_model", dis, (n5, r5), 128)[0] and not plan("run_model", dis, (n5, r5), 127)[0]
    # geometry-only (sigma-only, disentangled, tensor cores) reads the normalised planes only, with or without provenance
    geo = (False, True, (True, False), ("run_model", "single-gather"))
    assert plan("run_model", dis, (n5, r5), 256, sigma_only=True) == geo
    assert plan("run_model", dis, (n5, other), 256, sigma_only=True) == geo
    assert plan("run_model", dis, (n5, r5), 256, sigma_only=True, nfe_precision="fp32") == (False, False, (True, True), ("run_model", "two-gather"))

    # training: the identity needs the autograd sources of a registered pair, in the grad state it was registered in
    raw_t = torch.randn(2, 96, 4, 4, requires_grad=True)
    mean, std = torch.zeros(2, 96, 1, 1, requires_grad=True), torch.ones(2, 96, 1, 1, requires_grad=True)
    norm_t = raw_t * 1.0
    reg.provenance_put(raw_t, norm_t, std.detach().reshape(2, -1) + 1e-8, mean.detach().reshape(2, -1))
    reg.provenance_attach(raw_t, std, 1e-8, mean)
    pair = (norm_t.view(2, 3, 32, 4, 4), raw_t.view(2, 3, 32, 4, 4))
    p = field_plan("render", dis, *pair, opts, 2, 64, True)
    assert p.sources[0] is std and p.sources[1] is mean and p.path == ("render", "training-single-gather") and not p.stage_denorm
    assert torch.equal(p.affine[0], std.detach().reshape(2, 96) + 1e-8) and torch.equal(p.affine[1], mean.detach().reshape(2, 96))
    assert field_plan("run_model", dis, *pair, opts, 2, 256, True).path is None          # training run_model counts nothing
    refused = (False, False, (True, True), ("render", "training"))
    assert plan("render", dis, (pair[0].detach(), pair[1]), 64, grad=True) == refused   # norm detached after registration
    assert plan("render", dis, (pair[0], pair[1].detach()), 64, grad=True) == refused   # planes carry no grad
    # geometry-only in training still stages the raw planes unless the identity applies: the backward returns their gradient
    assert plan("run_model", dis, pair, 256, grad=True, sigma_only=True) == (True, True, (True, False), None)
    assert plan("run_model", dis, (pair[0].detach(), pair[1]), 256, grad=True, sigma_only=True) == (False, True, (True, True), None)
    monkeypatch.setenv("NFE_BWD_LIBRARY_GEMM", "1")
    p = field_plan("render", dis, *pair, opts, 2, 64, True)
    assert p.affine is None and p.sources is None and p.library_gemm and p.path == ("render", "training")
    reg.clear()


def test_missing_library_fails_loudly(monkeypatch):
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/libnfe_b200.so")
    with pytest.raises(RuntimeError, match="not built"):
        _lib.load()


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "nerffaceediting_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src.replace("the CPU reference is the oracle", "").replace("(SURVEY.md §7.5, oracle nfo_resample_ray)", "") \
                    .replace("the oracle does not have", ""), f"{f} mentions the oracle"
                assert "_torch_render" not in src, f"{f} mentions the tests' torch restatement"


def test_decoder_recognition_by_structure():
    from nerffaceediting_b200 import triplane
    o = {'decoder_lr_mul': 1, 'decoder_output_dim': 32, 'decoder_seg_dim': 15}
    assert ops.describe_decoder(triplane.OSGDecoder(32, o))[0] == ops.DEC_OSG
    assert ops.describe_decoder(triplane.DisentangledOSGDecoder(32, o))[0] == ops.DEC_DISENTANGLED
    assert ops.describe_decoder(triplane.SegmentationOSGDecoder(32, o))[0] == ops.DEC_SEGMENTATION
    assert ops.describe_decoder(torch.nn.Linear(3, 3)) is None
    odd = triplane.OSGDecoder(32, dict(o, decoder_output_dim=16))
    assert ops.describe_decoder(odd) is None                                   # unsupported width -> staged path
    relu = triplane.OSGDecoder(32, o)
    relu.net[1] = torch.nn.ReLU()
    assert ops.describe_decoder(relu) is None
    # parameter names are the reference's (state dicts are interchangeable)
    assert sorted(triplane.DisentangledOSGDecoder(32, o).state_dict()) == sorted(
        f"{n}.{i}.{p}" for n in ("geo_net", "app_net") for i in (0, 2) for p in ("weight", "bias"))
    fc = triplane.FullyConnectedLayer(32, 64, lr_multiplier=0.5)
    assert abs(fc.weight_gain - 0.5 / np.sqrt(32)) < 1e-12 and fc.bias_gain == 0.5


def test_reference_decoder_state_dicts_load_into_recognised_decoders():
    """The state dicts of the reference's OSGDecoder, DisentangledOSGDecoder and SegmentationOSGDecoder (tests/golden/decoders.npz,
    recorded from the reference's modules) load strictly into this package's classes, which describe_decoder recognises."""
    from nerffaceediting_b200 import triplane
    g = np.load(os.path.join(ROOT, "tests", "golden", "decoders.npz"))
    for prefix, cls, kind in (("osg_lr1", triplane.OSGDecoder, ops.DEC_OSG), ("dis_lr1", triplane.DisentangledOSGDecoder, ops.DEC_DISENTANGLED),
                              ("seg_lr1", triplane.SegmentationOSGDecoder, ops.DEC_SEGMENTATION)):
        sd = {k[len(prefix) + 1:]: torch.from_numpy(g[k]) for k in g.files if k.startswith(prefix + ".") and ".out." not in k}
        assert sd
        dec = cls(32, {'decoder_lr_mul': 1, 'decoder_output_dim': 32, 'decoder_seg_dim': 15})
        dec.load_state_dict(sd, strict=True)
        assert ops.describe_decoder(dec)[0] == kind, prefix


@needs_reference
def test_reference_decoders_are_recognised_and_shadow_package_resolves():
    code = r"""
import sys, pickle
import training.triplane as t
from training.volumetric_rendering import renderer, ray_marcher, ray_sampler, math_utils
from nerffaceediting_b200 import ops
assert renderer.__file__.startswith(sys.argv[1]), renderer.__file__
assert t.__file__.startswith(sys.argv[2]), t.__file__
assert t.DisentangledImportanceRenderer is renderer.DisentangledImportanceRenderer
assert t.RaySampler is ray_sampler.RaySampler
o = {'decoder_lr_mul': 1, 'decoder_output_dim': 32, 'decoder_seg_dim': 15}
assert ops.describe_decoder(t.OSGDecoder(32, o))[0] == ops.DEC_OSG
assert ops.describe_decoder(t.DisentangledOSGDecoder(32, o))[0] == ops.DEC_DISENTANGLED
assert ops.describe_decoder(t.SegmentationOSGDecoder(32, o))[0] == ops.DEC_SEGMENTATION
r = pickle.loads(pickle.dumps(renderer.DisentangledImportanceRenderer()))
assert type(r).__module__ == 'training.volumetric_rendering.renderer'
assert type(r.ray_marcher).__module__ == 'training.volumetric_rendering.ray_marcher'
assert hasattr(math_utils, 'get_ray_limits_box') and hasattr(renderer, 'sample_from_3dgrid')
print('ok')
"""
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([os.path.join(ROOT, "shadow"), REFERENCE]))
    r = subprocess.run([sys.executable, "-c", code, os.path.join(ROOT, "shadow"), REFERENCE], capture_output=True, text=True, env=env)
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr[-2000:]


def test_synthetic_inputs():
    a = synth.hash_normal(3, (4, 5))
    assert a.dtype == np.float32 and np.array_equal(a, synth.hash_normal(3, (4, 5))) and not np.array_equal(a, synth.hash_normal(4, (4, 5)))
    big = synth.hash_normal(1, (200000,))
    assert abs(big.mean()) < 0.01 and abs(big.std() - 1) < 0.01
    c2w, k = synth.camera_sweep(8)
    assert c2w.shape == (8, 4, 4) and k.shape == (8, 3, 3)
    assert torch.allclose(c2w[:, :3, 3].norm(dim=-1), torch.full((8,), 2.7), atol=1e-5)
    assert abs(float(k[0, 0, 0]) - 4.2634) < 1e-3          # FOV 18.837 deg with the reference's 3.14159 / 1.414


def test_synth_cameras_are_the_stored_ones():
    """tests/golden/rays.npz stores the cameras whose rays the reference's RaySampler produced for the fixture; synth_inputs must
    still make exactly those cameras (look-at poses, 18.837 and 60 degree intrinsics)."""
    import math
    g = np.load(os.path.join(ROOT, "tests", "golden", "rays.npz"))
    c2w = synth.look_at_cam2world([math.pi / 2 - 0.4, math.pi / 2, math.pi / 2 + 0.3], [math.pi / 2 - 0.25, math.pi / 2, math.pi / 2 + 0.2])
    assert np.array_equal(c2w.numpy(), g["cam2world"])
    assert np.array_equal(synth.fov_to_intrinsics(18.837).numpy(), g["intrinsics"][0])
    assert np.array_equal(synth.fov_to_intrinsics(60.0).numpy(), g["intrinsics_wide"][0])


@needs_reference
def test_synth_cameras_match_reference_camera_utils():
    code = r"""
import sys, math, torch
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[2])
import camera_utils
import synth_inputs as synth
for h, v in ((math.pi/2, math.pi/2), (math.pi/2 - 0.4, math.pi/2 + 0.25)):
    ref = camera_utils.LookAtPoseSampler.sample(h, v, torch.tensor([0, 0, 0.2]), radius=2.7)
    assert torch.equal(ref, synth.look_at_cam2world([h], [v]))
assert torch.equal(camera_utils.FOV_to_intrinsics(18.837), synth.fov_to_intrinsics(18.837))
print('ok')
"""
    r = subprocess.run([sys.executable, "-c", code, ROOT, REFERENCE], capture_output=True, text=True)
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr[-2000:]


def test_state_dict_names_are_the_reference_s():
    """Checkpoints of the reference load unchanged: same parameter / buffer names and shapes (recorded from the reference's modules)."""
    from nerffaceediting_b200 import networks as net
    import os
    import sys
    import numpy as np
    here = os.path.dirname(os.path.abspath(__file__))
    sys.path.insert(0, os.path.join(here, "golden"))
    import conv_cases as cases
    g = np.load(os.path.join(here, "golden", "conv_stack.npz"))

    def keys(m):
        return sorted(f"{k}:{'x'.join(map(str, v.shape))}" for k, v in m.state_dict().items())
    assert keys(cases.make_synthesis(net)) == sorted(g["keys.synthesis"].tolist())
    assert keys(cases.make_mapping(net)) == sorted(g["keys.mapping"].tolist())
    assert keys(cases.make_sr(net, '2X')) == sorted(g["keys.sr2x"].tolist())
    assert keys(cases.make_sr(net, '8XDC')) == sorted(g["keys.sr8xdc"].tolist())
    assert keys(net.SuperresolutionHybrid4X(32, 256, 4, True)) == sorted(g["keys.sr4x"].tolist())
    assert keys(net.SuperresolutionHybrid8X(32, 512, 4, True)) == sorted(g["keys.sr8x"].tolist())


def test_modconv_plan_and_argument_checks_run_on_the_host(built):
    """nfe_modconv_workspace_bytes is pure host code (tile plan of conv_gemm_kernel): the struct layout the ctypes mirror assumes, the
    scratch sizes of known layers and the rejected configurations, without a GPU (SURVEY.md §8f row f3)."""
    lib = _lib.load()
    A = _lib.NfeModconvArgs
    assert A.noise_batch_stride.offset == 4 * 8 and A.fh.offset == 8 * 8 and A.weight_batch_stride.offset == 8 * 8 + 16 * 4      # 8 pointer-sized + 16 x 4 bytes
    assert ctypes.sizeof(A) == 8 * 8 + 16 * 4 + 8

    def need(**kw):
        base = dict(batch=8, in_ch=256, out_ch=256, in_h=256, in_w=256, ksize=3, up=1, demodulate=1, flip_weight=1, act=3, alpha=0.2, gain=1.0,
                    clamp=256.0, dtype=1)
        base.update(kw)
        return lib.nfe_modconv_workspace_bytes(A(**base))
    up256 = lambda v: (v + 255) // 256 * 256                                                                          # noqa: E731
    coef = up256((8 * 256 + 256 + 8) * 4)
    # fp16, plain 3x3: per item 9 taps x 256 x 256 halves of packed weights
    assert need() == coef + up256(8 * 9 * 256 * 256 * 2)
    assert need(out_ch=384) > 0                                      # three tiles of 128
    # fp32: hi + lo parts
    assert need(dtype=0) == coef + up256(8 * 9 * 256 * 256 * 2 * 2)
    # up = 2: the same nine taps + the (2H+1)^2 intermediate in the activation type
    assert need(up=2, in_h=128, in_w=128) == coef + up256(8 * 9 * 256 * 256 * 2) + up256(8 * 257 * 257 * 256 * 2)
    # 1x1 to 3 channels (ToRGB): the output tile is padded to 16 rows
    assert need(ksize=1, out_ch=3, demodulate=0) == up256((8 * 3 + 3 + 8) * 4) + up256(8 * 16 * 256 * 2)
    for bad in (dict(in_ch=24), dict(ksize=5), dict(up=2, ksize=1), dict(up=3), dict(dtype=2), dict(out_ch=400), dict(batch=0)):
        assert need(**bad) == -1, bad
        assert lib.nfe_last_error()


def test_modconv_cta_plans_fit_the_sm(built):
    """The CTA plan of every layer shape of the reference's generator (and a sweep around them), read through the host-only hook
    nfe_debug_modconv_plan: shared memory within the 227 KB a CTA may have, a weight ring of at least two slots (three beside the
    persistent CTA's stage region), every tap in exactly one weight block, and the up = 2 blocks paired as DESIGN.md §3.6 says."""
    lib = _lib.load()
    A = _lib.NfeModconvArgs
    fn = lib.nfe_debug_modconv_plan
    fn.argtypes = [ctypes.POINTER(A), ctypes.POINTER(ctypes.c_int), ctypes.c_int]
    fn.restype = ctypes.c_int

    def plan(**kw):
        base = dict(batch=8, in_ch=256, out_ch=256, in_h=256, in_w=256, ksize=3, up=1, demodulate=1, flip_weight=1, act=3, alpha=0.2, gain=1.0,
                    clamp=256.0, dtype=1)
        base.update(kw)
        out = (ctypes.c_int * 26)()
        assert fn(A(**base), out, 26) == 0, (kw, lib.nfe_last_error())
        keys = "parts ma sa kg n_tile n_tiles kc chunks sb b_stage b_slot persist stage_bytes n_blk taps smem ctas_per_sm".split()
        d = dict(zip(keys, out[:17]))
        d["widths"] = [w for w in out[17:] if w]
        return d

    shapes = []
    for dtype in (0, 1):
        for res, ch in ((4, 512), (8, 512), (16, 512), (32, 512), (64, 512), (128, 256), (256, 128), (512, 64)):      # backbone / SR ladders
            shapes.append(dict(dtype=dtype, in_ch=ch, out_ch=ch, in_h=res, in_w=res))
            shapes.append(dict(dtype=dtype, in_ch=min(2 * ch, 512), out_ch=ch, in_h=max(res // 2, 2), in_w=max(res // 2, 2), up=2))
            shapes.append(dict(dtype=dtype, in_ch=ch, out_ch=96, in_h=res, in_w=res, ksize=1, demodulate=0))
        for extra in (dict(in_ch=32, out_ch=256, in_h=128, in_w=128, up=2), dict(in_ch=256, out_ch=128, in_h=256, in_w=256, up=2),
                      dict(in_ch=16, out_ch=8, in_h=5, in_w=7), dict(in_ch=96, out_ch=40, in_h=33, in_w=9), dict(in_ch=64, out_ch=384, in_h=8, in_w=24),
                      dict(in_ch=48, out_ch=112, in_h=12, in_w=20, batch=1), dict(in_ch=2048, out_ch=256, in_h=64, in_w=64)):
            shapes.append(dict(dtype=dtype, **extra))
    seen_persist = seen_twin = seen_pairs = 0
    for kw in shapes:
        p = plan(**kw)
        assert p["smem"] <= 227 * 1024, (kw, p)
        assert p["sb"] >= (3 if p["persist"] else 2), (kw, p)
        assert sum(p["widths"]) == p["taps"] and len(p["widths"]) == p["n_blk"], (kw, p)
        assert p["b_slot"] == max(p["widths"]) * p["b_stage"], (kw, p)
        assert p["b_stage"] == p["parts"] * p["n_tile"] * p["kc"] * 2 and p["chunks"] * p["kc"] == kw["in_ch"], (kw, p)
        assert p["n_tile"] % 16 == 0 and p["n_tile"] * p["n_tiles"] >= kw["out_ch"], (kw, p)
        n_acc = 4 if kw.get("up", 1) == 2 else p["ma"]
        assert n_acc * p["n_tile"] <= 512, (kw, p)                                       # tensor-memory columns of one accumulator set
        if p["ctas_per_sm"] == 2 and p["ma"] == 1 and p["n_tile"] <= 128 and kw.get("up", 1) == 1 and kw.get("ksize", 3) == 3:
            assert 2 * (p["smem"] + 1024) <= 228 * 1024 and 2 * p["n_tile"] <= 512, (kw, p)      # twin CTAs really fit twice
            seen_twin += 1
        if kw.get("up", 1) == 2 and 2 * p["n_tile"] <= 256:
            assert p["widths"] == [2, 1, 2, 1, 2, 1], (kw, p)                            # (0,0)+(0,1) | (0,2) | (1,0)+(1,1) | (1,2) | (2,0)+(2,1) | (2,2)
            seen_pairs += 1
        elif kw.get("up", 1) == 1:
            assert p["widths"] == [1] * p["taps"], (kw, p)
        seen_persist += p["persist"]
    assert seen_persist and seen_twin and seen_pairs


def test_generator_state_dict_names_are_the_reference_s():
    """The whole-generator mirror (BASELINE configs[1]) accepts the reference's checkpoints: names and shapes recorded from the
    reference's TriPlaneGenerator (tests/golden/make_golden_generator.py)."""
    import numpy as np
    here = os.path.dirname(os.path.abspath(__file__))
    sys.path.insert(0, os.path.join(here, "golden"))
    import conv_cases as cases
    from nerffaceediting_b200 import triplane
    g = np.load(os.path.join(here, "golden", "generator.npz"))
    for which in cases.GENERATORS:
        G = cases.make_generator(triplane.TriPlaneGenerator, which)
        keys = sorted(f"{k}:{'x'.join(map(str, v.shape))}" for k, v in G.state_dict().items())
        assert keys == sorted(g[f"keys.{which}"].tolist())


@needs_reference
def test_shadow_torch_utils_resolves_and_delegates_cpu_calls():
    """shadow/torch_utils: bias_act / upfirdn2d / conv2d_resample come from the shadow, the rest of torch_utils from the reference; CPU
    tensors go through the reference's own functions, so a reference generator still runs on CPU with the shadow on the path."""
    code = r"""
import sys, torch
import training.networks_stylegan2 as ns
from torch_utils.ops import bias_act, upfirdn2d, conv2d_resample, fma, conv2d_gradfix
assert bias_act.__file__.startswith(sys.argv[1]) and conv2d_resample.__file__.startswith(sys.argv[1]) and upfirdn2d.__file__.startswith(sys.argv[1])
assert fma.__file__.startswith(sys.argv[2]) and conv2d_gradfix.__file__.startswith(sys.argv[2])
assert ns.bias_act is bias_act and ns.conv2d_resample is conv2d_resample and ns.upfirdn2d is upfirdn2d
torch.manual_seed(0)
block = ns.SynthesisBlock(16, 16, w_dim=8, resolution=8, img_channels=3, is_last=True).eval()
x, img, ws = torch.randn(2, 16, 4, 4), torch.randn(2, 3, 4, 4), torch.randn(2, 3, 8)
with torch.no_grad():
    y, im = block(x, img, ws, noise_mode='const')
assert y.shape == (2, 16, 8, 8) and im.shape == (2, 3, 8, 8) and torch.isfinite(im).all()
print('ok')
"""
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([os.path.join(ROOT, "shadow"), REFERENCE]))
    r = subprocess.run([sys.executable, "-c", code, os.path.join(ROOT, "shadow"), REFERENCE], capture_output=True, text=True, env=env)
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr[-2000:]
