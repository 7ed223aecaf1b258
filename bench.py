#!/usr/bin/env python
"""bench.py -- rays/sec of the SDF volume-rendering hot path (BASELINE.json metric), one workload per invocation.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--precision bf16x3|bf16|fp32]
                  [--dump-outputs DIR]

--dump-outputs DIR: after the timed steps, rank 0 writes what the timed path returned in its last timed step as DIR/<name>.npy
          (float32; at most 64 MB in all).  Inputs and parameters are seeded, so two builds run with the same arguments can be compared
          output for output.  Render workloads: the arrays SDFField.render returns (rgb, depth, normal, accumulation, bg_transmittance,
          weights).  angelo-train-8192: the loss and a fixed, seeded sample of every parameter after the optimizer step.  k_field_tc adds
          the per-warp partial sums of a ray in shared memory with atomics (S > 32), so the rendered values of two runs may differ in
          the last bits: compare with a tolerance.

Workloads (BASELINE.json configs; the default is the headline the metric is quoted on):
  neus-facto-dtu65-4096x128   configs[1]: DTU-scan65-shaped rays, 4096 rays x 128 samples per GPU, neus-facto SDFField (hash L=16 F=2
                              T=2^19, geo MLP 71-256-256-257, colour MLP 321-256-256-3).  One step = UniformSampler(128) ->
                              SDFField.get_outputs -> alpha weights -> RGB / depth / normal / accumulation, i.e. the render pass of
                              SurfaceModel.get_outputs (models/base_surface_model.py:292-365): ONE fused launch (field + compositing).
  volsdf-errorbounded-4096    configs[2]: same scene / field shape, ErrorBoundedSampler (64 + 32 extra samples, up to 5 x 128-sample
                              refinements, 10 bisection steps) with the Laplace density, density-form weights (models/volsdf.py:62-87).
  bakedsdf-render-65536       configs[4]: contracted scene, off-axis PE (deg 8), ref-nerf heads; ProposalNetworkSampler (256, 96) -> 48
                              samples; 65 536 rays per step per GPU, render only.
  angelo-train-8192           configs[3]: neus-facto-angelo training step (numerical gradients, hash F=8) at 8192 rays per GPU with the
                              gradient all-reduce over NCCL inside the timed region.

training_step (headline line only): the angelo-train-8192 step measured at the same N in child processes (one per rank, own NCCL
          rendezvous): train rays/s with the DistributedDataParallel gradient all-reduce inside the timed region, `allreduce_alone_ms`.
value   : whole-job rays/s, inputs resident in HBM, CUDA-event time (max over ranks), L2 flushed between steps.
e2e     : same metric through the public module API with HOST (pinned) ray buffers: H2D of the rays and D2H of the rendered
          rgb / depth / normal / accumulation inside the timed region (the headline workload replays one CUDA graph per step).
roofline: the dominant kernel against the measured peak of MEASURED_PEAKS.json (burst peak: the kernel is event-timed alone).
cpu_baseline / --impl reference: the CPU oracle port (oracle/, a restatement of the reference's torch-CPU path, pinned to the
          unmodified reference by tests/golden) on a bounded sample of the same workload, all host threads.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

R_PER_GPU, S = 4096, 128
FLOP_PER_SAMPLE = 763904     # SURVEY.md section 8d: 381 952 MAC (geo 149 504 + grad 83 968 + colour 148 480)
FLOP_PER_SDF_EVAL = 299008   # geo network only (149 504 MAC): what the samplers' sdf_fn costs
FLOP_PER_SAMPLE_BAKED = 1071616  # SURVEY.md section 8d config 5: 535 808 MAC
WORKLOAD = "neus-facto-dtu65-4096x128"
WORKLOADS = (WORKLOAD, "volsdf-errorbounded-4096", "bakedsdf-render-65536", "angelo-train-8192")
AABB = [[-1.0, -1, -1], [1, 1, 1]]
VOLSDF_BETA = 0.01   # Laplace beta of the volsdf workload: small like a trained scene, so that the error-bounded refinement loop actually iterates
DUMP_BYTES = 64_000_000


def dump_outputs(out_dir, arrays):
    """Writes {name: tensor} as out_dir/<name>.npy in float32 (float64 stays float64)."""
    import numpy as np

    arrs = {k: v.detach().cpu().to(torch.float64 if v.dtype == torch.float64 else torch.float32).numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrs.values())
    if total > DUMP_BYTES:
        raise ValueError(f"--dump-outputs: {total} bytes exceed the {DUMP_BYTES} byte budget")
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrs.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), a)


# ------------------------------------------------------------------------------------------------------------------ fields
def make_field(device, precision="fp32", seed=0, table_dtype="fp32", beta_init=0.3):
    """The product SDFField of the headline workload (neus-facto preset, method_configs.py:472-480 + README override
    inside_outside=False), random-init + perturbation so that hash + PE inputs matter."""
    import sdfstudio_b200 as sb
    from sdfstudio_b200.synthetic import perturb_field_

    torch.manual_seed(seed)
    cfg = sb.SDFFieldConfig(use_grid_feature=True, num_layers=2, num_layers_color=2, hidden_dim=256, bias=0.5, beta_init=beta_init,
                            use_appearance_embedding=False, inside_outside=False, grid_layout="torch", precision=precision, table_dtype=table_dtype)
    field = sb.SDFField(cfg, torch.tensor(AABB), num_images=49)
    perturb_field_(field, seed)
    return field.to(device).eval()


def make_baked_field(device, precision="bf16x3", seed=0):
    """bakedsdf-shaped field (method_configs.py:265-292): L-inf contraction, off-axis PE degree 8, diffuse / tint / reflections / n.v."""
    import sdfstudio_b200 as sb
    from sdfstudio_b200.synthetic import perturb_field_

    class _Contraction:
        order = float("inf")

    torch.manual_seed(seed)
    cfg = sb.SDFFieldConfig(use_grid_feature=True, num_layers=2, num_layers_color=2, hidden_dim=256, bias=0.05, beta_init=0.1, inside_outside=False,
                            position_encoding_max_degree=8, use_diffuse_color=True, use_specular_tint=True, use_reflections=True, use_n_dot_v=True,
                            off_axis=True, grid_layout="torch", precision=precision)
    field = sb.SDFField(cfg, torch.tensor(AABB), num_images=49, spatial_distortion=_Contraction())
    perturb_field_(field, seed)
    return field.to(device).eval()


def oracle_of(field, spec=None):
    """CPU oracle holding the SAME parameters as `field` (cpu_baseline / reference arm only)."""
    from oracle.field import FieldSpec, OracleField

    if spec is None:
        spec = FieldSpec(num_layers=2, num_layers_color=2, hidden_dim=256, use_grid_feature=True, grid_layout="torch")
    sd = {k: v.detach().cpu() for k, v in field.state_dict().items()}
    sd["hash_table"] = sd.pop("encoding.hash_table")
    return OracleField(spec, sd)


def read_traffic(workload, precision):
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel from the committed `ncu --set full` capture."""
    for name in (f"r02_ncu_{workload}_{precision}_summary.json", f"r02_ncu_field_tc_{precision}_summary.json"):
        p = os.path.join(ROOT, "profiles", name)
        if not os.path.exists(p):
            continue
        try:
            with open(p) as fh:
                d = json.load(fh)

            def mb(k):
                v, u = float(d[k]["value"]), d[k]["unit"]
                return v * {"Mbyte": 1e6, "Gbyte": 1e9, "Kbyte": 1e3, "byte": 1.0}[u]
            return mb("dram__bytes_read.sum") + mb("dram__bytes_write.sum")
        except Exception:  # noqa: BLE001
            return None
    return None


def read_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as fh:
            d = json.load(fh)
        return {"bf16_tflops": d.get("bf16_tflops", 1590.0), "bf16_tflops_sustained": d.get("bf16_tflops_sustained", 1400.0),
                "hbm_gbs": d.get("hbm_gbs", 6650.0), "source": "measured"}
    return {"bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "hbm_gbs": 6650.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md clocks line)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.gpu_index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(smax) if smax else None, "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------------ CPU arm
def oracle_step(oracle, o, d, cam, nears, fars, S_):
    """The headline step on the CPU through the oracle port (what the reference's torch-CPU path computes)."""
    from oracle import render, samplers

    b = samplers.spaced_sampler(nears, fars, S_, "uniform")
    out = oracle.get_outputs(o, d, b.starts, b.deltas, cam, return_alphas=True)
    w, _ = samplers.weights_from_alphas(out["alphas"][..., 0])
    w = w[..., None]
    rgb = render.render_rgb(out["rgb"], w, torch.ones(3))
    depth = render.render_depth(w, b.starts[..., None], b.ends[..., None], "expected")
    normal = render.render_semantics(out["normals"], w)
    acc = render.render_accumulation(w)
    return rgb, depth, normal, acc


def oracle_step_volsdf(oracle, o, d, cam, nears, fars):
    """models/volsdf.py:62-87 on the CPU: ErrorBoundedSampler (sdf_fn = the oracle's geo network) -> field -> density weights -> renderers."""
    from oracle import render, samplers

    sdf_fn = lambda starts: oracle.get_sdf(o, d, starts)  # noqa: E731
    b = samplers.error_bounded_sampler(nears, fars, sdf_fn, oracle.get_beta())
    b = b[0] if isinstance(b, tuple) else b
    out = oracle.get_outputs(o, d, b.starts, b.deltas, cam)
    w, _ = samplers.weights_from_density(b.deltas, out["density"][..., 0])
    w = w[..., None]
    return (render.render_rgb(out["rgb"], w, torch.ones(3)), render.render_depth(w, b.starts[..., None], b.ends[..., None], "expected"),
            render.render_semantics(out["normals"], w), render.render_accumulation(w))


def cpu_arm(workload, rays_per_step, steps, warmup):
    """rays/s of the CPU oracle port on the host cores (best thread count <= all cores), bounded sample of the workload."""
    from sdfstudio_b200.synthetic import dtu_like_rays

    ncpu = os.cpu_count() or 1
    o, d, cam, nears, fars = dtu_like_rays(rays_per_step, 4242)
    if workload == "bakedsdf-render-65536":
        from oracle.field import FieldSpec

        spec = FieldSpec(num_layers=2, num_layers_color=2, hidden_dim=256, use_grid_feature=True, position_encoding_max_degree=8, use_diffuse_color=True,
                         use_specular_tint=True, use_reflections=True, use_n_dot_v=True, off_axis=True, contraction="linf", grid_layout="torch")
        oracle = oracle_of(make_baked_field("cpu", "fp32"), spec)
        nears, fars = torch.full_like(nears, 0.2), torch.full_like(fars, 6.0)
        fn = lambda: oracle_step(oracle, o, d, cam, nears, fars, 48)  # noqa: E731  (field + compositing at the 48 final samples)
    elif workload == "volsdf-errorbounded-4096":
        oracle = oracle_of(make_field("cpu", beta_init=VOLSDF_BETA))
        fn = lambda: oracle_step_volsdf(oracle, o, d, cam, nears, fars)  # noqa: E731
    else:
        oracle = oracle_of(make_field("cpu"))
        fn = lambda: oracle_step(oracle, o, d, cam, nears, fars, S)  # noqa: E731
    # torch-CPU does not scale monotonically with threads: pick the fastest thread count <= all cores (one timed step each)
    best, cores = None, ncpu
    for t in sorted({min(ncpu, c) for c in (16, 32, 64, ncpu)}):
        torch.set_num_threads(t)
        if rays_per_step <= 256:
            fn()
        t0 = time.perf_counter()
        fn()
        dt = time.perf_counter() - t0
        if best is None or dt < best:
            best, cores = dt, t
    torch.set_num_threads(cores)
    for _ in range(warmup):
        fn()
    t0 = time.perf_counter()
    for _ in range(steps):
        fn()
    dt = (time.perf_counter() - t0) / max(steps, 1)
    return rays_per_step / dt, dt, cores


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.workload == "angelo-train-8192":
        print(json.dumps({"impl": "reference", "unavailable": "the oracle port has no training step (autograd through the reference's modules is the reference itself, which cannot travel to the GPU box)"}))
        return
    # the headline workload runs its FULL 4096-ray batch per step (about 2 s of CPU work each); the heavier steps use a bounded sample
    full = args.workload == WORKLOAD
    rays = R_PER_GPU if full else 256
    warm = max(min(args.warmup, 3), 1) if not full else 1
    steps = args.steps
    value, dt, cores = cpu_arm(args.workload, rays, steps, warm)
    sample = f"{rays} rays per step ({'the full batch' if full else 'bounded sample'}) of the {args.workload} step ({dt * 1e3:.0f} ms/step), {steps} steps after {warm} warm-up"
    line = {
        "impl": "reference", "metric": "rays/sec at 4096 rays x 128 samples" if full else f"rays/sec, {args.workload}", "value": value, "unit": "rays/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": {"workload": args.workload, "sample": sample, "host_threads": cores, "host_cores_available": os.cpu_count()},
        "cpu_baseline": {"value": value, "unit": "rays/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }  # fmt: skip
    print(json.dumps(line))


def train_section(world, rank, steps=5, warmup=3, timeout=300):
    """BASELINE.json configs[3] next to the headline: every rank runs tools/train_workload.py (8192 rays per GPU, DistributedDataParallel gradient
    all-reduce over NCCL inside the timed region) in a child process on its own GPU with its own rendezvous (MASTER_PORT + 17), so that the
    driver's 1/2/4/8-GPU runs of this file also measure the one collective of the path.  Isolated on purpose: a failure or a hang of the
    training step cannot take the headline measurement down (the child is killed after `timeout` seconds and the section reports the error)."""
    import subprocess

    env = dict(os.environ)
    env.pop("TORCHELASTIC_USE_AGENT_STORE", None)          # the child's rank 0 hosts its own store
    env.pop("TORCHELASTIC_RUN_ID", None)
    if world > 1:
        env["MASTER_PORT"] = str(int(env.get("MASTER_PORT", "29500")) + 17)
    cmd = [sys.executable, os.path.join(ROOT, "tools", "train_workload.py"), "--steps", str(steps), "--warmup", str(warmup)]
    try:
        p = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=timeout)
    except subprocess.TimeoutExpired:
        return {"workload": "angelo-train-8192", "error": f"timed out after {timeout} s"}
    if rank != 0:
        return None
    lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
    if p.returncode != 0 or not lines:
        return {"workload": "angelo-train-8192", "error": (p.stderr or p.stdout).strip().splitlines()[-1][:300] if (p.stderr or p.stdout).strip() else f"exit code {p.returncode}"}
    t = json.loads(lines[-1])
    return {"workload": "angelo-train-8192", "metric": t["metric"], "value": t["value"], "unit": t["unit"], "n_gpus": t["n_gpus"], "steps": t["steps"], "warmup": t["warmup"],
            "ms_per_step": t["ms_per_step"], "scaling": "weak", "rays_per_gpu": t["config"]["rays_per_gpu"], "parallelism": t["config"]["parallelism"],
            "gradient_bytes": t["config"]["gradient_bytes"], "allreduce_alone_ms": t["config"]["allreduce_alone_ms"], "e2e": t["e2e"], "gpu_launches": t["gpu_launches"],
            "roofline": t["roofline"], "loss": t["loss"]}


# ------------------------------------------------------------------------------------------------------------------ GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=WORKLOAD, choices=WORKLOADS)
    ap.add_argument("--precision", default=os.environ.get("SDFB200_PRECISION", "auto"))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--unfused", action="store_true", help="A/B: separate field and compositing launches (per-sample heads through HBM)")
    ap.add_argument("--no-graph", action="store_true", help="A/B: e2e without CUDA-graph replay")
    ap.add_argument("--no-train-section", action="store_true", help="skip the training-step section (angelo-train-8192 with the NCCL gradient all-reduce) of the headline line")
    ap.add_argument("--table-dtype", default="fp32", choices=["fp32", "fp16"], help="fp16 = gather from a half-precision copy (tiny-cuda-nn's storage)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        return run_reference(args)
    if args.workload == "angelo-train-8192":
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import train_workload

        return train_workload.main(args)

    import torch.distributed as dist

    import sdfstudio_b200 as sb
    from sdfstudio_b200.synthetic import dtu_like_rays

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU path in the product)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    precision = args.precision
    if precision == "auto":
        precision = "bf16x3"   # tcgen05 path at parity-grade precision (bf16 split, fp32 accumulate); fp32 / bf16 via --precision
    wl = args.workload
    white = torch.ones(3, device=dev)
    H = sb.FieldHeadNames
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    field_ms = []
    extra = {}

    # ---- per-workload modules, rays (ray shard of this rank: independent rays, no data-path collective; SURVEY section 8e) and step ----
    if wl == WORKLOAD:
        R = R_PER_GPU
        field = make_field(dev, precision, table_dtype=args.table_dtype)
        sampler = sb.UniformSampler(num_samples=S).eval()
        o, d, cam, nears, fars = dtu_like_rays(R, 1000 + rank)

        def step(o_, d_, n_, f_, time_field=False):
            rb = sb.RayBundle(origins=o_, directions=d_, pixel_area=pix, directions_norm=pix, camera_indices=cam_d, nears=n_, fars=f_)
            rs = sampler(rb)
            if time_field:
                e0, e1 = ev(), ev()
                e0.record()
            if args.unfused:
                out = field(rs, return_alphas=True)
                res = None
            else:
                res = field.render(rs, white)          # field + compositing: one fused launch (+ the global depth clip)
            if time_field:
                e1.record()
                field_ms.append((e0, e1))
            return res if res is not None else sb.render_from_alphas(out[H.ALPHA], out[H.RGB], out[H.NORMAL], rs, white)

        flop_per_launch = FLOP_PER_SAMPLE * R * S
        cfg = {"workload": wl, "rays_per_gpu": R, "samples_per_ray": S, "sampler": "UniformSampler(128), eval",
               "field": f"neus-facto SDFField L16 F2 T2^19 MLP 2x256 (torch-layout table, {args.table_dtype})", "precision": precision,
               "step": "separate field + compositing launches" if args.unfused else "SDFField.render: field + compositing fused in k_field_tc"}
        kernel = "k_field_tc (sdfb200_field_render)" if precision != "fp32" else "sdfb200_field_forward (k_sgemm + elementwise kernels)"
        cpu_sample = 256
    elif wl == "volsdf-errorbounded-4096":
        R = R_PER_GPU
        field = make_field(dev, precision, table_dtype=args.table_dtype, beta_init=VOLSDF_BETA)   # SURVEY 8d config 3: LaplaceDensity(beta_init=0.1); 0.01 = a trained-scene beta
        sampler = sb.ErrorBoundedSampler(num_samples=64, num_samples_eval=128, num_samples_extra=32, eps=0.1, beta_iters=10, max_total_iters=5).eval()
        o, d, cam, nears, fars = dtu_like_rays(R, 1000 + rank)
        counters = {"sdf_points": 0, "calls": 0}

        def sdf_fn(rs):
            counters["sdf_points"] += rs.frustums.starts.shape[0] * rs.frustums.starts.shape[1]
            counters["calls"] += 1
            return field.get_sdf(rs)

        def step(o_, d_, n_, f_, time_field=False):
            rb = sb.RayBundle(origins=o_, directions=d_, pixel_area=pix, directions_norm=pix, camera_indices=cam_d, nears=n_, fars=f_)
            if time_field:
                e0, e1 = ev(), ev()
                e0.record()
            rs, _ = sampler(rb, density_fn=field.laplace_density, sdf_fn=sdf_fn)
            res = field.render(rs, white, from_density=True)
            if time_field:
                e1.record()
                field_ms.append((e0, e1))
            return res

        flop_per_launch = None   # filled from the measured number of sdf evaluations
        cfg = {"workload": wl, "rays_per_gpu": R, "sampler": "ErrorBoundedSampler(64, eval 128, extra 32, eps 0.1, 10 bisections, <= 5 rounds), eval",
               "field": f"neus-facto-shaped SDFField L16 F2 T2^19 MLP 2x256 + LaplaceDensity ({args.table_dtype} table)", "precision": precision,
               "step": "sampler (sdf-only k_field_tc passes + per-ray scans) -> SDFField.render(from_density) (96 samples: 128 % 96 != 0 -> field kernel + compositing kernels)"}
        kernel = "whole step: k_field_tc sdf-only passes (sampler) + field pass + sampler scans"
        cpu_sample = 64
    else:  # bakedsdf-render-65536
        R = 65536
        field = make_baked_field(dev, precision)
        aabb = torch.tensor(AABB)
        g = torch.Generator().manual_seed(1)

        class _Contraction:
            order = float("inf")

        nets = []
        for max_res in (64, 256):   # bakedsdf.py proposal networks: hidden 16, 5 levels, log2 T 17
            f = sb.HashMLPDensityField(aabb, num_layers=2, hidden_dim=16, spatial_distortion=_Contraction(), num_levels=5, max_res=max_res,
                                       log2_hashmap_size=17).to(dev).eval()
            with torch.no_grad():
                nb = f.mlp_base
                nb.params[nb.n_net:] = ((torch.rand(nb.n_grid, generator=g) * 2 - 1) * 2.0).to(dev)
            nets.append(f)
        fns = [n.density_fn for n in nets]
        sampler = sb.ProposalNetworkSampler(num_proposal_samples_per_ray=(256, 96), num_nerf_samples_per_ray=48, num_proposal_network_iterations=2,
                                            use_uniform_sampler=False).eval()
        o, d, cam, nears, fars = dtu_like_rays(R, 1000 + rank)
        nears, fars = torch.full_like(nears, 0.2), torch.full_like(fars, 1000.0)   # method_configs.py:275-276

        def step(o_, d_, n_, f_, time_field=False):
            rb = sb.RayBundle(origins=o_, directions=d_, pixel_area=pix, directions_norm=pix, camera_indices=cam_d, nears=n_, fars=f_)
            rs, _, _ = sampler(rb, density_fns=fns)
            if time_field:
                e0, e1 = ev(), ev()
                e0.record()
            res = field.render(rs, white)
            if time_field:
                e1.record()
                field_ms.append((e0, e1))
            return res

        flop_per_launch = FLOP_PER_SAMPLE_BAKED * R * 48
        cfg = {"workload": wl, "rays_per_gpu": R, "samples_per_ray": 48, "sampler": "ProposalNetworkSampler(256, 96 -> 48), 2 HashMLPDensityFields, eval",
               "field": "bakedsdf SDFField: L-inf contraction, off-axis PE deg 8 (371-wide input), diffuse / tint / reflections / n.v, L16 F2 T2^19", "precision": precision,
               "step": "proposal sampler -> SDFField.render (generic engine: per-layer tcgen05 Linear kernels + compositing kernels)"}
        kernel = "sdfb200_field_render (k_tc_linear x layers + elementwise + k_render_alphas)"
        cpu_sample = 64

    cfg["l2"] = "flushed between timed steps (256 MiB write)"
    cfg["parallelism"] = f"ray-shard x{world}, no data-path collective (rendering shards over rays; the gradient all-reduce lives in the training workload)"
    host = [t.pin_memory() for t in (o, d, nears, fars)]
    cam_d = cam.view(-1, 1).to(dev)
    pix = torch.ones(R, 1, device=dev)
    dev_in = [t.to(dev) for t in host]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.no_grad():
        for _ in range(max(args.warmup, 3)):
            step(*dev_in)
        barrier()
        if wl == "volsdf-errorbounded-4096":
            counters["sdf_points"], counters["calls"] = 0, 0
        launches0 = sb._lib.launch_count()
        clocks = ClockSampler(local_rank)
        if rank == 0:
            clocks.start()
        # ---- device-resident timing ----
        pairs = []
        barrier()
        for _ in range(args.steps):
            flush.zero_()
            e0, e1 = ev(), ev()
            e0.record()
            last = step(*dev_in, time_field=True)
            e1.record()
            pairs.append((e0, e1))
        barrier()
        launches = sb._lib.launch_count() - launches0
        dev_ms = sum(a.elapsed_time(b) for a, b in pairs)
        fld_ms = sum(a.elapsed_time(b) for a, b in field_ms)
        if wl == "volsdf-errorbounded-4096":
            extra["sdf_evals_per_ray"] = counters["sdf_points"] / (R * args.steps)
            extra["sdf_fn_calls_per_step"] = counters["calls"] / args.steps
            flop_per_launch = FLOP_PER_SDF_EVAL * counters["sdf_points"] / args.steps + FLOP_PER_SAMPLE * R * 96
        # ---- spot check of what was just timed: the exact-fp32 CUDA-core engine on a strided subset of the same rays ----
        if precision != "fp32" and wl == WORKLOAD:
            chk = make_field(dev, "fp32", table_dtype=args.table_dtype)
            sub = torch.arange(0, R, 64, device=dev)
            rb_s = sb.RayBundle(origins=dev_in[0][sub], directions=dev_in[1][sub], pixel_area=pix[sub], directions_norm=pix[sub], camera_indices=cam_d[sub],
                                nears=dev_in[2][sub], fars=dev_in[3][sub])
            ref = chk.render(sampler(rb_s), white)
            extra["check_vs_fp32_engine"] = {"rays": int(sub.numel()), "max_abs_rgb": float((ref["rgb"] - last["rgb"][sub]).abs().max()),
                                             "max_rel_depth": float(((ref["depth"] - last["depth"][sub]).abs() / ref["depth"].abs().clamp_min(1e-3)).max())}
            del chk
        # ---- end-to-end timing: host rays in, rendered images out ----
        out_host = {k: torch.empty(s, dtype=torch.float32).pin_memory() for k, s in (("rgb", (R, 3)), ("depth", (R, 1)), ("normal", (R, 3)), ("accumulation", (R, 1)))}
        graph = None
        static_in = [torch.empty_like(t) for t in dev_in]
        if wl == WORKLOAD and not args.no_graph:
            # capture sampler -> fused field + compositing -> depth clip once; every step = 4 H2D copies, one graph replay, 4 D2H copies
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):
                    step(*static_in)
            torch.cuda.current_stream().wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                static_out = step(*static_in)

        def e2e_step():
            for dst, src in zip(static_in, host):
                dst.copy_(src, non_blocking=True)
            r = static_out if graph is not None else step(*static_in)
            if graph is not None:
                graph.replay()
            for k, t in out_host.items():
                t.copy_(r[k], non_blocking=True)

        for _ in range(3):
            e2e_step()
        barrier()
        pairs2 = []
        for _ in range(args.steps):
            flush.zero_()
            e0, e1 = ev(), ev()
            e0.record()
            e2e_step()
            e1.record()
            pairs2.append((e0, e1))
        barrier()
        e2e_ms = sum(a.elapsed_time(b) for a, b in pairs2)
        clk = clocks.stop() if rank == 0 else None

    # ---- the training step of the path (configs[3]) with its gradient all-reduce, measured next to the headline at the same N ----
    train = None
    if wl == WORKLOAD and not args.no_train_section:
        torch.cuda.empty_cache()
        train = train_section(world, rank, args.steps, args.warmup)
        barrier()
    times = torch.tensor([dev_ms, e2e_ms, fld_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms, fld_ms = (float(x) for x in times)
    if rank == 0:
        peaks = read_peaks()
        rays_total = R * world * args.steps
        value = rays_total / (dev_ms * 1e-3)
        e2e = rays_total / (e2e_ms * 1e-3)
        achieved_tflops = flop_per_launch / (fld_ms / args.steps * 1e-3) / 1e12
        h2d = sum(t.numel() * t.element_size() for t in host)
        d2h = sum(t.numel() * t.element_size() for t in out_host.values())
        cpu = None
        if not args.no_cpu_baseline:
            cv, cdt, cores = cpu_arm(wl, cpu_sample, 4, 1)
            cpu = {"value": cv, "unit": "rays/s", "cores": cores, "kind": "port", "sample": f"{cpu_sample} rays per step of the same step, 4 steps ({cdt*1e3:.0f} ms/step)"}
        cfg["e2e_path"] = "CUDA graph replay (sampler + fused field/compositing + depth clip) between pinned H2D / D2H copies" if graph is not None else "module calls between pinned H2D / D2H copies"
        line = {
            "metric": "rays/sec at 4096 rays x 128 samples" if wl == WORKLOAD else f"rays/sec, {wl}", "value": value, "unit": "rays/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": {"fp32": "f32", "bf16x3": "bf16x3 (fp32 accumulate)", "bf16": "bf16 (fp32 accumulate)"}[precision], "data": "synthetic",
            "config": cfg,
            "e2e": {"value": e2e, "unit": "rays/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": int(launches),
            "roofline": {"bound": "tensor", "achieved": achieved_tflops, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
                         "frac": achieved_tflops / peaks["bf16_tflops"], "traffic": read_traffic(wl, precision), "peak_source": peaks["source"] + " bf16_tflops (burst)",
                         "kernel": kernel, "ms_per_launch": fld_ms / args.steps, "algorithmic_flop_per_launch": flop_per_launch},
            "cpu_baseline": cpu, "clocks": clk,
        }  # fmt: skip
        line.update(extra)
        if train is not None:
            line["training_step"] = train
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {k: v for k, v in last.items() if isinstance(v, torch.Tensor)})
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
