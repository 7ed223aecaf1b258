"""bench.py --workload angelo-train-8192 (BASELINE.json configs[3]): one TRAINING step of the neus-facto-angelo field
(method_configs.py:404-432: hash L=16 F=8 T=2^22 base 64 max 4096, linear interpolation, one hidden geo layer 167-256-257, colour MLP 4x256,
numerical gradients = 7 geo evaluations per sample, PE zeroed, appearance embedding, progressive level mask) at 8192 rays per GPU:

    ProposalNetworkSampler (256, 96 -> 48 samples, two HashMLPDensityFields, no grad) -> SDFField training forward (tcgen05 GEMMs of
    linear_ops.py + this package's twice-differentiable grid operator) -> alpha compositing -> rgb L1 + eikonal + curvature-free loss
    -> backward -> gradient all-reduce over NCCL (DistributedDataParallel, the reference's own wrapper: pipelines/base_pipeline.py:241-243)
    -> Adam.

The all-reduce is INSIDE the timed region (it is part of loss.backward() under DDP).  value = train rays/s over all ranks (weak scaling:
8192 rays per GPU).  The line also carries the stand-alone cost of an all-reduce of the same gradient bytes (`allreduce_alone_ms`) so the
bounding collective is visible, and the HBM roofline of the hash-grid traffic (gathers forward + scatter-adds backward).
"""
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

R_TRAIN, S_TRAIN = 8192, 48


def make_angelo_field(dev, precision, log2_t=22, seed=0):
    import sdfstudio_b200 as sb
    from sdfstudio_b200.synthetic import perturb_field_

    torch.manual_seed(seed)
    cfg = sb.SDFFieldConfig(use_grid_feature=True, num_layers=1, num_layers_color=4, hidden_dim=256, hidden_dim_color=256, geo_feat_dim=256, bias=0.5,
                            beta_init=0.3, inside_outside=False, use_appearance_embedding=True, use_numerical_gradients=True, base_res=64, max_res=4096,
                            num_levels=16, log2_hashmap_size=log2_t, hash_features_per_level=8, hash_smoothstep=False, use_position_encoding=False,
                            grid_layout="torch", precision=precision)
    field = sb.SDFField(cfg, torch.tensor([[-1.0, -1, -1], [1, 1, 1]]), num_images=49)
    perturb_field_(field, seed)
    field.update_mask(8)                         # progressive training starts at level_init = 8 (method_configs.py:425-427)
    field.set_numerical_gradients_delta(1.0 / 4096.0)
    return field.to(dev).train()


def main(args):
    import torch.distributed as dist
    from torch.nn.parallel import DistributedDataParallel as DDP

    import bench
    import sdfstudio_b200 as sb
    from sdfstudio_b200.synthetic import dtu_like_rays

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    precision = "bf16x3" if args.precision == "auto" else args.precision
    torch.backends.cuda.matmul.allow_tf32 = True           # scripts/train.py:59 (only the small ATen leftovers are affected)
    field = make_angelo_field(dev, precision)
    aabb = torch.tensor([[-1.0, -1, -1], [1, 1, 1]])
    g = torch.Generator().manual_seed(1)
    nets = []
    for max_res in (64, 256):
        f = sb.HashMLPDensityField(aabb, num_layers=2, hidden_dim=16, num_levels=5, max_res=max_res, log2_hashmap_size=17).to(dev).eval()
        with torch.no_grad():
            nb = f.mlp_base
            nb.params[nb.n_net:] = ((torch.rand(nb.n_grid, generator=g) * 2 - 1) * 2.0).to(dev)
        nets.append(f)
    fns = [n.density_fn for n in nets]
    sampler = sb.ProposalNetworkSampler(num_proposal_samples_per_ray=(256, 96), num_nerf_samples_per_ray=S_TRAIN, num_proposal_network_iterations=2,
                                        use_uniform_sampler=False).train()

    class Step(torch.nn.Module):
        """field + compositing + loss as ONE module so that DDP sees every parameter of the step"""

        def __init__(self, field):
            super().__init__()
            self.field = field

        def forward(self, rs, target, white):
            fo = self.field(rs, return_alphas=True)
            out = sb.render_from_alphas(fo[sb.FieldHeadNames.ALPHA], fo[sb.FieldHeadNames.RGB], fo[sb.FieldHeadNames.NORMAL], rs, white, training=True)
            eik = ((fo[sb.FieldHeadNames.GRADIENT].norm(2, dim=-1) - 1) ** 2).mean()
            return (out["rgb"] - target).abs().mean() + 0.1 * eik

    model = Step(field)
    if world > 1:
        model = DDP(model, device_ids=[local_rank], find_unused_parameters=True, gradient_as_bucket_view=True)
    params = [p for p in model.parameters() if p.requires_grad]
    opt = torch.optim.Adam(params, lr=5e-4, eps=1e-15, fused=True)   # AdamOptimizerConfig(lr, eps) of method_configs.py:404-432; single-pass (fused) implementation
    R = R_TRAIN
    o, d, cam, nears, fars = dtu_like_rays(R, 2000 + rank)
    host = [t.pin_memory() for t in (o, d, nears, fars)]
    dev_in = [t.to(dev) for t in host]
    cam_d = cam.view(-1, 1).to(dev)
    pix = torch.ones(R, 1, device=dev)
    target = torch.rand(R, 3, device=dev)
    white = torch.ones(3, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def step(o_, d_, n_, f_):
        rb = sb.RayBundle(origins=o_, directions=d_, pixel_area=pix, directions_norm=pix, camera_indices=cam_d, nears=n_, fars=f_)
        with torch.no_grad():
            rs, _, _ = sampler(rb, density_fns=fns)
        loss = model(rs, target, white)
        opt.zero_grad(set_to_none=True)
        loss.backward()                                    # under DDP: gradient all-reduce (NCCL) overlapped / finished in here
        opt.step()
        return loss.detach()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    for _ in range(max(args.warmup, 3)):
        step(*dev_in)
    barrier()
    launches0 = sb._lib.launch_count()
    clocks = bench.ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    pairs = []
    barrier()
    for _ in range(args.steps):
        flush.zero_()
        e0, e1 = ev(), ev()
        e0.record()
        loss = step(*dev_in)
        e1.record()
        pairs.append((e0, e1))
    barrier()
    launches = sb._lib.launch_count() - launches0
    dev_ms = sum(a.elapsed_time(b) for a, b in pairs)
    if args.dump_outputs and rank == 0:
        # the loss and a fixed, seeded sample (<= 65536 entries) of every parameter as the last timed step left them
        g_dump = torch.Generator().manual_seed(0)
        dumped = {"loss": loss.clone()}
        for name, p in field.named_parameters():
            flat = p.detach().reshape(-1)
            idx = torch.randint(0, flat.numel(), (65536,), generator=g_dump).sort().values if flat.numel() > 65536 else torch.arange(flat.numel())
            dumped["param." + name] = flat[idx.to(dev)].clone()
    # end to end: host rays in, scalar loss out (the reference's train_iteration returns the loss dict to the host: trainer.py:319-327)
    loss_host = torch.empty((), dtype=torch.float32).pin_memory()
    pairs2 = []
    for _ in range(args.steps):
        flush.zero_()
        e0, e1 = ev(), ev()
        e0.record()
        loss = step(*[t.to(dev, non_blocking=True) for t in host])
        loss_host.copy_(loss, non_blocking=True)
        e1.record()
        pairs2.append((e0, e1))
    barrier()
    e2e_ms = sum(a.elapsed_time(b) for a, b in pairs2)
    # the collective alone: one all-reduce of the same gradient bytes
    n_grad = sum(p.numel() for p in params)
    ar_ms = None
    if world > 1:
        buf = torch.empty(n_grad, device=dev, dtype=torch.float32)
        for _ in range(2):
            dist.all_reduce(buf)
        barrier()
        e0, e1 = ev(), ev()
        e0.record()
        for _ in range(3):
            dist.all_reduce(buf)
        e1.record()
        torch.cuda.synchronize()
        ar_ms = e0.elapsed_time(e1) / 3
        del buf
    clk = clocks.stop() if rank == 0 else None
    times = torch.tensor([dev_ms, e2e_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms = (float(x) for x in times)
    if rank == 0:
        peaks = bench.read_peaks()
        rays_total = R * world * args.steps
        ms = dev_ms / args.steps
        n_samples = R * S_TRAIN
        active = 8 / 16.0                                                   # level mask at level_init = 8
        table_bytes = 2 * 7 * 16 * 8 * 32 * active * n_samples              # forward gathers + backward scatter-adds, F = 8 fp32 rows of 32 B
        achieved = table_bytes / (ms * 1e-3) / 1e9
        line = {
            "metric": "train rays/sec, angelo-train-8192", "value": rays_total / (dev_ms * 1e-3), "unit": "rays/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": f"{precision} GEMMs (fp32 accumulate), fp32 table / optimizer", "data": "synthetic",
            "config": {"workload": "angelo-train-8192", "rays_per_gpu": R, "samples_per_ray": S_TRAIN,
                       "field": "neus-facto-angelo SDFField: hash L16 F8 T2^22 (2.1 GB fp32), geo 167-256-257, colour 4x256, numerical gradients (7 geo evaluations / sample), level mask 8/16",
                       "step": "proposal sampler (no grad) -> field fwd (tcgen05 GEMMs + grid operator) -> compositing -> L1 + eikonal -> backward -> all-reduce -> Adam",
                       "parallelism": f"data parallel x{world}: ray shard per rank, DistributedDataParallel gradient all-reduce over NCCL inside the timed region",
                       "gradient_bytes": n_grad * 4, "allreduce_alone_ms": ar_ms, "l2": "flushed between timed steps (256 MiB write)"},
            "e2e": {"value": rays_total / (e2e_ms * 1e-3), "unit": "rays/s", "h2d_bytes_per_step": sum(t.numel() * 4 for t in host), "d2h_bytes_per_step": 4},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"], "traffic": None,
                         "peak_source": peaks["source"] + " hbm_gbs", "kernel": "hash-grid operator (k_grid_encode forward gathers + k_grid_encode_bwd scatter-adds) over the whole step",
                         "algorithmic_bytes_per_step": table_bytes},
            "cpu_baseline": None, "clocks": clk, "loss": float(loss),
        }
        if args.dump_outputs:
            bench.dump_outputs(args.dump_outputs, dumped)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    # stand-alone entry (bench.py's headline workload spawns it once per rank to attach the training step to its line)
    import argparse

    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--precision", default="auto")
    ap.add_argument("--dump-outputs", metavar="DIR")
    main(ap.parse_args())
