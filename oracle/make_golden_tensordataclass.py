"""TEST INFRASTRUCTURE -- mints tests/golden/reference_tensordataclass.json from the UNMODIFIED reference: the dataclass fields of
RayBundle / RaySamples / Frustums (cameras/rays.py:233-339), the FieldHeadNames values, and the exact memory layout (shape, stride,
storage offset, shared storages and their contents) of the RaySamples the reference's UniformSampler returns for a seeded [H, W]
camera bundle.  tests/test_abi_cpu.py rebuilds objects with that structure and layout and runs the product's host-side accessors on them.

    python -m oracle.make_golden_tensordataclass
"""
import dataclasses
import json
import os

import torch

from . import ref_import

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "reference_tensordataclass.json")
H, W, S, SEED = 5, 7, 9, 2


def camera_bundle_inputs():
    """The seeded [H, W] camera ray bundle fields (shared with the test that replays the fixture)."""
    g = torch.Generator().manual_seed(SEED)
    d = torch.randn(H, W, 3, generator=g)
    d = d / d.norm(dim=-1, keepdim=True)
    return dict(origins=torch.randn(H, W, 3, generator=g), directions=d, pixel_area=torch.ones(H, W, 1), directions_norm=torch.ones(H, W, 1),
                camera_indices=torch.zeros(H, W, 1, dtype=torch.long), nears=torch.full((H, W, 1), 0.5), fars=torch.full((H, W, 1), 4.5))


def fields_of(cls):
    return [[f.name, f.default is dataclasses.MISSING and f.default_factory is dataclasses.MISSING] for f in dataclasses.fields(cls)]


def layout(tensors):
    """{name: shape / stride / offset / storage index} plus the distinct storages (dtype + flat contents) they view."""
    storages, keys, out = [], {}, {}
    for name, t in tensors.items():
        st = t.untyped_storage()
        key = (st.data_ptr(), t.dtype)
        if key not in keys:
            keys[key] = len(storages)
            flat = torch.empty(0, dtype=t.dtype).set_(st)
            storages.append({"dtype": str(t.dtype).replace("torch.", ""), "data": flat.tolist()})
        out[name] = {"shape": list(t.shape), "stride": list(t.stride()), "offset": t.storage_offset(), "storage": keys[key]}
    return out, storages


def main():
    ref = ref_import.ref_modules()
    bundle = ref.RayBundle(**camera_bundle_inputs())
    flat = bundle.flatten()
    rs = ref.ray_samplers.UniformSampler(num_samples=S).eval()(flat)
    fr = rs.frustums
    tensors = {f"frustums.{n}": getattr(fr, n) for n in ("origins", "directions", "starts", "ends", "pixel_area")}
    tensors.update({n: getattr(rs, n) for n in ("camera_indices", "deltas", "spacing_starts", "spacing_ends")})
    views, storages = layout(tensors)
    fixture = {"RayBundle": fields_of(ref.RayBundle), "RaySamples": fields_of(ref.RaySamples), "Frustums": fields_of(ref.Frustums),
               "FieldHeadNames": {h.name: h.value for h in ref.FieldHeadNames}, "sampler": f"UniformSampler(num_samples={S}).eval()",
               "ray_samples": views, "storages": storages}
    with open(OUT, "w") as fh:
        json.dump(fixture, fh, indent=1, sort_keys=True)
    print("wrote", OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    main()
