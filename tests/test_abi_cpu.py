"""CPU-only: the C-ABI library builds/loads, exports every symbol include/sdfb200.h declares, and the ctypes struct
mirrors have the library's sizes.  No compute calls (no GPU here)."""
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    src = open(os.path.join(ROOT, "include", "sdfb200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(sdfb200_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from sdfstudio_b200 import _lib

    lib = _lib.load()
    syms = header_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/sdfb200.h but not exported"
    # and the python binding knows each of them
    assert set(syms) == set(_lib.EXPORTED_SYMBOLS), set(syms) ^ set(_lib.EXPORTED_SYMBOLS)
    assert lib.sdfb200_version() == 100


def test_struct_sizes_match():
    import ctypes as C

    from sdfstudio_b200 import _lib

    lib = _lib.load()
    for which, st in enumerate((_lib.GridDesc, _lib.FieldDesc, _lib.FieldParams, _lib.FieldIn, _lib.FieldOut, _lib.RenderOut, _lib.FieldRender)):
        assert lib.sdfb200_struct_size(which) == C.sizeof(st)


def test_invalid_arguments_return_error_codes_not_crashes():
    import sdfstudio_b200 as sb
    from sdfstudio_b200 import _lib

    lib = _lib.load()
    g = _lib.GridDesc()
    g.n_levels = 99  # > MAX
    assert lib.sdfb200_grid_encode(g, None, None, 4, None, 0, None, None) == -1
    assert b"n_levels" in lib.sdfb200_last_error_string()
    with pytest.raises(_lib.Sdfb200Error):
        _lib.check(lib.sdfb200_spaced_bins(None, None, None, None, 0, 4, 0, 0, None, None, None))
    # unsupported field shapes are refused at plan time
    d = _lib.FieldDesc()
    assert lib.sdfb200_field_packed_bytes(d) == 0


def test_field_descriptor_roundtrip_all_presets():
    """packed / workspace size queries succeed for the five BASELINE config shapes (host logic only)."""
    import torch

    import sdfstudio_b200 as sb
    from sdfstudio_b200 import _lib

    lib = _lib.load()
    aabb = torch.tensor([[-1.0, -1, -1], [1, 1, 1]])
    presets = {
        "neus-facto": dict(use_grid_feature=True, num_layers=2, num_layers_color=2, log2_hashmap_size=12),
        "volsdf": dict(num_layers=8, num_layers_color=4),
        "angelo": dict(use_grid_feature=True, num_layers=1, num_layers_color=4, use_numerical_gradients=True, hash_features_per_level=8,
                       hash_smoothstep=False, use_position_encoding=False, log2_hashmap_size=12, base_res=64, max_res=4096),
        "bakedsdf": dict(use_grid_feature=True, num_layers=2, num_layers_color=2, position_encoding_max_degree=8, use_diffuse_color=True,
                         use_specular_tint=True, use_reflections=True, use_n_dot_v=True, off_axis=True, log2_hashmap_size=12),
    }
    for name, kw in presets.items():
        f = sb.SDFField(sb.SDFFieldConfig(**kw), aabb, 4)
        d = f._field_desc()
        assert lib.sdfb200_field_packed_bytes(d) > 0, name
        assert lib.sdfb200_field_workspace_bytes(d, 1000) > 0, name
    # state-dict names follow the reference (SURVEY appendix A.2)
    names = set(dict(sb.SDFField(sb.SDFFieldConfig(**presets["neus-facto"]), aabb, 4).named_parameters()))
    for n in ("glin0.weight_g", "glin0.weight_v", "glin2.bias", "clin0.weight_v", "laplace_density.beta", "deviation_network.variance",
              "embedding_appearance.embedding.weight", "encoding.params"):
        assert n in names, n


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "sdfstudio_b200")
    for dirpath, _, files in os.walk(pkg):
        for fn in files:
            if fn.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, fn)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, flags=re.M), f"{fn} imports oracle"
                assert "oracle/" not in txt and "oracle." not in txt.replace("oracle.make_golden", ""), f"{fn} references oracle"


# ---------------------------------------------------------------------------------------------------------------
# checkpoint compatibility (SURVEY.md 8f row 4): same state_dict names and shapes as the unmodified reference SDFField
# (fixture minted by oracle/make_golden_statedict.py), and the trainer's checkpoint layout loads
# ---------------------------------------------------------------------------------------------------------------
def _product_field_cpu(name, layout="tcnn"):
    import json

    import sdfstudio_b200 as sb
    from oracle import cases

    spec, kw = cases.CASES[name]
    cfg = sb.SDFFieldConfig(
        num_layers=spec.num_layers, hidden_dim=spec.hidden_dim, geo_feat_dim=spec.geo_feat_dim, num_layers_color=spec.num_layers_color,
        hidden_dim_color=spec.hidden_dim_color, appearance_embedding_dim=spec.appearance_embedding_dim,
        use_appearance_embedding=spec.use_appearance_embedding, use_grid_feature=spec.use_grid_feature,
        position_encoding_max_degree=spec.position_encoding_max_degree, use_diffuse_color=spec.use_diffuse_color,
        use_specular_tint=spec.use_specular_tint, use_reflections=spec.use_reflections, use_n_dot_v=spec.use_n_dot_v, off_axis=spec.off_axis,
        use_numerical_gradients=spec.use_numerical_gradients, num_levels=spec.num_levels, max_res=spec.max_res, base_res=spec.base_res,
        log2_hashmap_size=min(spec.log2_hashmap_size, 12), hash_features_per_level=spec.hash_features_per_level, hash_smoothstep=spec.hash_smoothstep,
        use_position_encoding=spec.use_position_encoding, grid_layout=layout)  # fmt: skip
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "sdffield_state_keys.json")) as fh:
        ref = json.load(fh)[name]
    return sb.SDFField(cfg, torch.tensor([[-1.0, -1, -1], [1, 1, 1]]), num_images=49), ref


@pytest.mark.parametrize("name", ["neusfacto_c1", "angelo_small", "bakedsdf_small", "volsdf_stock"])
def test_state_dict_names_match_reference(name):
    field, ref = _product_field_cpu(name)
    mine = {k: list(v.shape) for k, v in field.state_dict().items() if not k.startswith("encoding.")}
    assert mine == ref
    assert [k for k in field.state_dict() if k.startswith("encoding.")] == ["encoding.params"]      # tcnn's single flat vector


def test_reference_checkpoint_layout_loads():
    from sdfstudio_b200 import checkpoint

    src, _ = _product_field_cpu("neusfacto_c1")
    dst, _ = _product_field_cpu("neusfacto_c1")
    g = torch.Generator().manual_seed(3)
    with torch.no_grad():
        for p in src.parameters():
            p.copy_(torch.randn(p.shape, generator=g))
    # what engine/trainer.py:276-297 writes for a DDP-wrapped pipeline, with tcnn's fp16 grid parameters
    pipe = {"module._model.field." + k: (v.half() if k == "encoding.params" else v.clone()) for k, v in src.state_dict().items()}
    pipe["module._model.proposal_networks.0.mlp_base.params"] = torch.zeros(7)
    pipe["module.datamanager.train_camera_optimizer.pose_adjustment"] = torch.zeros(3, 6)
    ckpt = {"step": 1000, "pipeline": pipe, "optimizers": {}, "schedulers": {}, "scalers": {}}
    missing, unexpected = checkpoint.load_field_checkpoint(dst, ckpt)
    assert not missing and not unexpected
    for (k, a), (_, b) in zip(src.state_dict().items(), dst.state_dict().items()):
        assert torch.equal(a.half().float() if k == "encoding.params" else a, b), k
    torch_layout, _ = _product_field_cpu("neusfacto_c1", layout="torch")
    with pytest.raises(ValueError):
        checkpoint.load_field_checkpoint(torch_layout, ckpt)


# ---------------------------------------------------------------------------------------------------------------
# the Python mirrors keep the reference's constructor signatures and config defaults (fixture minted from the unmodified
# reference by oracle/make_golden_api.py)
# ---------------------------------------------------------------------------------------------------------------
def test_mirror_signatures_and_config_defaults_match_reference():
    import dataclasses
    import inspect
    import json

    import sdfstudio_b200 as sb

    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_api.json")) as fh:
        ref = json.load(fh)

    def plain(v):
        if isinstance(v, (int, float, str, bool)) or v is None:
            return v
        if isinstance(v, (tuple, list)):
            return [plain(x) for x in v]
        return f"<{type(v).__name__}>"

    mine_cfg = {f.name: plain(f.default) for f in dataclasses.fields(sb.SDFFieldConfig) if f.name != "_target" and f.default is not dataclasses.MISSING}
    b200_knobs = {"grid_layout", "precision", "table_dtype", "train_gemm"}
    assert {k: v for k, v in mine_cfg.items() if k not in b200_knobs} == ref["SDFFieldConfig"]
    problems = []
    for name, sig in ref.items():
        if name == "SDFFieldConfig":
            continue
        cls = getattr(sb, name, None) or getattr(sb.sdf_field, name, None)
        assert cls is not None, f"{name} is not mirrored"
        params = [(n, p) for n, p in inspect.signature(cls.__init__).parameters.items() if n not in ("self", "kwargs", "args")]
        mine = [[n, None if p.default is inspect.Parameter.empty else plain(p.default)] for n, p in params]
        # every reference parameter exists, in the same order, with the same default (extra trailing B200 keyword arguments are allowed)
        if mine[: len(sig)] != sig:
            problems.append((name, mine[: len(sig)], sig))
    assert not problems, problems


def test_spaced_sampler_accepts_the_reference_callables():
    import sdfstudio_b200 as sb
    from sdfstudio_b200.ray_samplers import identify_spacing

    # the lambdas exactly as the reference's subclasses write them (ray_samplers.py:130-247)
    assert identify_spacing(lambda x: x, lambda x: x) == "uniform"
    assert identify_spacing(lambda x: 1 / x, lambda x: 1 / x) == "lindisp"
    assert identify_spacing(torch.sqrt, lambda x: x**2) == "sqrt"
    assert identify_spacing(torch.log, torch.exp) == "log"
    assert identify_spacing(lambda x: torch.where(x < 1, x / 2, 1 - 1 / (2 * x)), lambda x: torch.where(x < 0.5, 2 * x, 1 / (2 - 2 * x))) == "piecewise"
    s = sb.SpacedSampler(spacing_fn=torch.sqrt, spacing_fn_inv=lambda x: x**2, num_samples=8)
    assert s.spacing == "sqrt" and s.num_samples == 8
    assert sb.UniformLinDispPiecewiseSampler(num_samples=4).spacing == "piecewise"
    with pytest.raises(NotImplementedError):
        sb.SpacedSampler(spacing_fn=lambda x: x**3, spacing_fn_inv=lambda x: x ** (1 / 3))
    with pytest.raises(ValueError):
        sb.SpacedSampler(spacing_fn=torch.sqrt, spacing_fn_inv=lambda x: x)


def test_proposal_network_checkpoint_layout_loads():
    """neus-facto / bakedsdf proposal networks (fields/density_fields.py:89-96): `mlp_base.params` of a trainer checkpoint loads; the MLP
    part has tiny-cuda-nn's element count (output layer padded to 16 neurons)."""
    import sdfstudio_b200 as sb
    from sdfstudio_b200 import checkpoint

    aabb = torch.tensor([[-1.0, -1, -1], [1, 1, 1]])
    src = sb.HashMLPDensityField(aabb, num_layers=2, hidden_dim=16, num_levels=5, max_res=64, log2_hashmap_size=12)
    dst = sb.HashMLPDensityField(aabb, num_layers=2, hidden_dim=16, num_levels=5, max_res=64, log2_hashmap_size=12)
    nb = src.mlp_base
    assert nb.n_net == 16 * 16 + 16 * 16          # FullyFusedMLP(n_neurons 16, 1 hidden layer): [16, pad16(10)] + [16 (padded output), 16]
    with torch.no_grad():
        nb.params.copy_(torch.randn(nb.params.shape, generator=torch.Generator().manual_seed(4)))
    ckpt = {"step": 1, "pipeline": {"module._model.proposal_networks.0.mlp_base.params": nb.params.detach().half(),      # tcnn stores fp16 or fp32
                                    "module._model.proposal_networks.0.aabb": aabb, "module._model.field.laplace_density.beta": torch.ones(1)}}
    checkpoint.load_density_field_checkpoint(dst, ckpt, index=0)
    assert torch.equal(dst.mlp_base.params.detach(), nb.params.detach().half().float())
    wrong = sb.HashMLPDensityField(aabb, num_layers=2, hidden_dim=16, num_levels=5, max_res=64, log2_hashmap_size=13)
    with pytest.raises(ValueError):
        checkpoint.load_density_field_checkpoint(wrong, ckpt, index=0)


def _reference_tensordataclasses():
    """(RayBundle class, RaySamples of the reference's UniformSampler, FieldHeadNames values) rebuilt from the fixture minted from the
    unmodified reference by oracle/make_golden_tensordataclass.py: classes with the reference's dataclass fields, and every tensor of the
    RaySamples with the reference's exact shape, stride, storage offset and storage sharing."""
    import dataclasses
    import json

    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_tensordataclass.json")) as fh:
        fx = json.load(fh)
    cls = {name: dataclasses.make_dataclass(name, [(f, object) if required else (f, object, dataclasses.field(default=None)) for f, required in fx[name]])
           for name in ("RayBundle", "RaySamples", "Frustums")}
    storages = [torch.tensor(s["data"], dtype=getattr(torch, s["dtype"])) for s in fx["storages"]]
    views = {name: storages[v["storage"]].as_strided(v["shape"], v["stride"], v["offset"]) for name, v in fx["ray_samples"].items()}
    frustums = cls["Frustums"](**{k.split(".", 1)[1]: v for k, v in views.items() if k.startswith("frustums.")})
    rs = cls["RaySamples"](frustums=frustums, **{k: v for k, v in views.items() if not k.startswith("frustums.")})
    for name, v in fx["ray_samples"].items():
        t = views[name]
        assert list(t.shape) == v["shape"] and list(t.stride()) == v["stride"] and t.storage_offset() == v["offset"], name
    return cls["RayBundle"], rs, fx["FieldHeadNames"]


def test_reference_tensordataclasses_pass_through_the_host_side():
    """The reference's own RayBundle / RaySamples (TensorDataclass objects with expanded stride-0 fields, cameras/rays.py:233-339) are what the
    modules receive inside sdfstudio: the host-side accessors must read them, keep their TYPE when slicing / flattening, and rebuild the
    [R, S+1] bin buffer the kernels take.  Structure only: no kernel runs."""
    from oracle.make_golden_tensordataclass import H, W, S, camera_bundle_inputs

    import sdfstudio_b200 as sb
    from sdfstudio_b200 import parallel

    RayBundle, rs, ref_heads = _reference_tensordataclasses()
    bundle = RayBundle(**camera_bundle_inputs())
    flat, hw = parallel.flatten_ray_bundle(bundle)
    assert hw == (H, W) and type(flat) is type(bundle) and flat.origins.shape == (H * W, 3) and flat.camera_indices.dtype == torch.long
    assert torch.equal(flat.origins.view(H, W, 3), bundle.origins)
    part = parallel.slice_ray_bundle(flat, 3, 11)
    assert type(part) is type(bundle) and part.origins.shape == (8, 3) and torch.equal(part.fars, flat.fars[3:11])
    sh = parallel.shard_ray_bundle(flat, 1, 3)
    assert sh.origins.shape[0] == parallel.shard_bounds(H * W, 1, 3)[1] - parallel.shard_bounds(H * W, 1, 3)[0]
    # the reference sampler's RaySamples of `flat`: starts / ends are overlapping slices of one bin buffer, origins / directions stride-0 expanded
    assert rs.frustums.origins.stride()[1] == 0 and rs.frustums.starts.untyped_storage().data_ptr() == rs.frustums.ends.untyped_storage().data_ptr()
    bins = sb.rays.bins_of(rs)
    assert bins.shape == (H * W, S + 1) and bins.is_contiguous()
    assert torch.equal(bins[:, :-1], rs.frustums.starts[..., 0]) and torch.equal(bins[:, 1:], rs.frustums.ends[..., 0])
    sp = sb.rays.spacing_bins_of(rs)
    assert torch.equal(sp[:, :-1], rs.spacing_starts[..., 0]) and torch.equal(sp[:, -1], rs.spacing_ends[:, -1, 0])
    o2, d2 = sb.rays.rays_of(rs)
    assert o2.is_contiguous() and torch.equal(o2, flat.origins) and torch.equal(d2, flat.directions)
    # FieldHeadNames of the reference compare equal to the product's keys (dicts returned by SDFField are indexed with either)
    assert set(ref_heads.values()) >= {h.value for h in sb.FieldHeadNames} or all(ref_heads[h.name] == h.value for h in sb.FieldHeadNames)


def test_grouped_grid_calls_reject_bad_groups_and_encoding_context_nests():
    """host logic of the grouped grid operator: argument validation of the C entry points (no launch) and the Encoding.point_groups context."""
    import sdfstudio_b200 as sb
    from sdfstudio_b200 import _lib

    lib = _lib.load()
    enc = sb.HashEncoding(num_levels=4, min_res=4, max_res=32, log2_hashmap_size=8, features_per_level=2)
    desc = enc._desc_ref()
    # n not a multiple of the group size / NULL pointers: error codes, not crashes
    assert lib.sdfb200_grid_encode_grouped(desc, None, None, 10, 7, None, 8, None) != 0
    assert lib.sdfb200_grid_encode_grouped(desc, None, None, 14, 7, None, 8, None) != 0
    assert lib.sdfb200_grid_encode_backward_grouped(desc, None, None, 14, 0, None, None) != 0
    assert lib.sdfb200_grid_encode_grouped(desc, None, None, 0, 7, None, 8, None) == 0          # empty batch
    assert enc._groups == 1
    with enc.point_groups(7):
        assert enc._groups == 7
        with enc.point_groups(6):
            assert enc._groups == 6
        assert enc._groups == 7
    assert enc._groups == 1


def test_bench_train_section_reports_child_failures(monkeypatch):
    """bench.py attaches the training step measured in child processes; a failing / hanging child must become an `error` entry of the
    section, never an exception of the headline measurement."""
    import subprocess
    import sys

    sys.path.insert(0, ROOT)
    import bench

    class R:
        returncode, stdout, stderr = 1, "", "Traceback ...\nRuntimeError: boom"

    monkeypatch.setattr(subprocess, "run", lambda *a, **k: R())
    out = bench.train_section(1, 0)
    assert out["workload"] == "angelo-train-8192" and "boom" in out["error"]

    def hang(*a, **k):
        raise subprocess.TimeoutExpired(cmd="x", timeout=1)

    monkeypatch.setattr(subprocess, "run", hang)
    assert "timed out" in bench.train_section(2, 0)["error"]

    class OK:
        returncode, stderr = 0, ""
        stdout = 'noise\n{"metric": "m", "value": 1.0, "unit": "rays/s", "n_gpus": 2, "steps": 5, "warmup": 3, "ms_per_step": 2.0, "config": {"rays_per_gpu": 8192, ' \
                 '"parallelism": "dp", "gradient_bytes": 4, "allreduce_alone_ms": 0.5}, "e2e": {}, "gpu_launches": 3, "roofline": {}, "loss": 0.1}\n'

    monkeypatch.setattr(subprocess, "run", lambda *a, **k: OK())
    sec = bench.train_section(2, 0)
    assert sec["value"] == 1.0 and sec["n_gpus"] == 2 and sec["allreduce_alone_ms"] == 0.5
    assert bench.train_section(2, 1) is None                                                   # only rank 0 reports
