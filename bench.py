#!/usr/bin/env python
"""Flagship benchmark: ResNet-50 DDP training step with the cgx comm hook
(bits=4, bucket_size=512) -- BASELINE.json configs[1] -- on N B200s of one node.

    python bench.py                                   # N=1, short
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 \
        --master-port 29500 bench.py --gpus 8 --steps 20 --warmup 5

One JSON line on rank 0 (contract in the task description):
  value          whole-job images/s, device-timed (CUDA events, max over ranks), inputs resident
  e2e.value      same step through the public API *including* the per-step H2D copy of the
                 batch from pinned host memory and the D2H read of the loss
  gpu_launches   launches of this repo's own fused allreduce kernel inside the timed region
Other models of BASELINE.json: --model gpt2-medium | vit-l16 (tokens/s or images/s).
--backend nccl runs the same script on stock NCCL DDP (same-box yardstick).
--impl reference would run the unmodified reference from baseline/_ref; it cannot be
installed on this image (needs OpenMPI: see DESIGN.md), so it reports `unavailable`.
--dump-outputs DIR saves the loss, gradients and weights of the last device-timed step as .npy
files; inputs are seeded and cuDNN runs deterministic convolutions, so for the ResNet models every
run with the same arguments computes the same values and two builds can be compared output for output.
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

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

# elements kept per array by --dump-outputs: two float32 arrays of 16 MB each
DUMP_SAMPLE = 1 << 22


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=20)
    p.add_argument("--warmup", type=int, default=5)
    p.add_argument("--impl", default="cgx", choices=["cgx", "reference"])
    p.add_argument("--backend", default="cgx", choices=["cgx", "nccl"])
    p.add_argument("--model", default="resnet50", choices=["resnet50", "resnet18", "gpt2-medium", "gpt2-small", "vit-l16", "vit-b16"])
    p.add_argument("--batch", type=int, default=0, help="per-GPU batch (0 = model default)")
    p.add_argument("--seq-len", type=int, default=1024)
    p.add_argument("--bits", type=int, default=-1, help="quantization bits (-1 = BASELINE config of the model)")
    p.add_argument("--bucket-size", type=int, default=512)
    p.add_argument("--layer-min-size", type=int, default=1024)
    p.add_argument("--stochastic", type=int, default=-1)
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-nccl-arm", action="store_true", help="skip the same-run NCCL DDP yardstick")
    p.add_argument("--no-allreduce", action="store_true", help="skip the allreduce micro-benchmark block (N > 1)")
    p.add_argument("--no-selftest", action="store_true", help="skip the multi-rank correctness self-test (N > 1)")
    p.add_argument("--hook", default="native", choices=["native", "python"],
                   help="native: C++ comm hook on the DDP reducer (default); python: cgx_hook as in the reference")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="write what the last device-timed step of the measured arm computed to DIR/<name>.npy: "
                        "loss.npy, grads.npy (the allreduced gradients) and params.npy (the updated weights); "
                        f"grads and params are the same seeded sample of {DUMP_SAMPLE} elements of the "
                        "flattened parameters when the model has more")
    args = p.parse_args()
    if args.steps < 1:
        p.error("--steps must be >= 1")
    return args


def last_step_outputs(params, loss):
    """The loss of a step, the gradients its allreduce delivered and the weights its optimizer
    wrote, as numpy arrays; gradients and weights are flattened in parameter order and reduced to
    the same fixed, seeded sample of DUMP_SAMPLE positions when there are more."""
    import torch

    params = list(params)
    grads = torch.cat([p.grad.detach().reshape(-1).float() for p in params])
    weights = torch.cat([p.detach().reshape(-1).float() for p in params])
    n = grads.numel()
    if n > DUMP_SAMPLE:
        idx = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE].sort().values
        idx = idx.to(grads.device)
        grads, weights = grads[idx], weights[idx]
    return {"loss": loss.detach().double().reshape(1).cpu().numpy(),
            "grads": grads.cpu().numpy(), "params": weights.cpu().numpy()}


MODEL_DEFAULTS = {
    # model: (per-GPU batch, bits, stochastic, metric unit)
    "resnet50": (128, 4, 0, "images/s"),
    "resnet18": (256, 4, 0, "images/s"),
    "gpt2-medium": (8, 8, 0, "tokens/s"),
    "gpt2-small": (16, 8, 0, "tokens/s"),
    "vit-l16": (32, 2, 1, "images/s"),
    "vit-b16": (64, 2, 1, "images/s"),
}


def reference_unavailable():
    why = "reference setup.py needs OpenMPI (ompi_info, -lmpi, mpi-ext.h); none in this image and no network -- see baseline/reference_install.log"
    ref = ROOT / "baseline" / "_ref"
    if ref.exists() and any(ref.glob("torch_cgx*.so")):
        why = "baseline/_ref has a build but it needs mpirun + CUDA-aware MPI at run time, not present on this image"
    print(json.dumps({"impl": "reference", "unavailable": why}))


def allreduce_microbench(dev, rank, world, nccl_pg, native):
    """Device-timed cgx {2,4,8,32}-bit allreduce vs ncclAllReduce at this N: back-to-back calls over
    rotating buffers (> 2x L2 in total), CUDA events, max over ranks, clocks sampled meanwhile."""
    import torch
    import torch.distributed as dist

    from torch_cgx_b200.utils.clocks import ClockSampler

    sampler = ClockSampler(dev.index)
    if rank == 0:
        sampler.start()
    saved = {k: os.environ.get(k) for k in ("CGX_COMPRESSION_QUANTIZATION_BITS", "CGX_COMPRESSION_BUCKET_SIZE")}
    os.environ["CGX_COMPRESSION_BUCKET_SIZE"] = "512"

    def timeit(fn, bufs, iters, warmup=3):
        for i in range(warmup):
            fn(bufs[i % len(bufs)])
        torch.cuda.synchronize()
        reps = []
        for _ in range(3):
            dist.barrier()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(iters):
                fn(bufs[i % len(bufs)])
            e1.record()
            torch.cuda.synchronize()
            reps.append(e0.elapsed_time(e1) * 1e3 / iters)
        t = torch.tensor(reps, device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return sorted(t.tolist())[1]

    rows = []
    try:
        for mb in (1, 16, 64, 256):
            nbytes = mb << 20
            n = nbytes // 4
            nbuf = max(2, min(16, (288 << 20) // nbytes + 1))
            bufs = [torch.randn(n, device=dev) for _ in range(nbuf)]
            iters = 20 if mb <= 64 else 6
            row = {"mb": mb, "dtype": "float32"}
            if nccl_pg is not None:
                row["nccl_us"] = round(timeit(lambda x: dist.all_reduce(x, group=nccl_pg), bufs, iters), 2)
            for bits in (2, 4, 8, 32):
                os.environ["CGX_COMPRESSION_QUANTIZATION_BITS"] = str(bits)
                for x in bufs:
                    x.normal_()
                native.reset_stats()
                t = timeit(lambda x: dist.all_reduce(x), bufs, iters)
                st = native.stats()
                row[f"cgx_{bits}bit_us"] = round(t, 2)
                row[f"cgx_{bits}bit_wire_gbs"] = round(st[3] / max(1, st[0]) / t / 1e3, 1)
                if "nccl_us" in row:
                    row[f"cgx_{bits}bit_vs_nccl"] = round(row["nccl_us"] / t, 3)
            rows.append(row)
            del bufs
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    return {"rows": rows, "clocks": sampler.stop() if rank == 0 else None,
            "timing": "CUDA events around back-to-back calls over rotating buffers (> 2x L2 in total), max over ranks, median of 3",
            "wire_gbs": "packed bytes this rank pushed over NVLink per call / time (per direction; 770 GB/s measured peer-copy peak)"}


def main():
    args = parse_args()
    if args.impl == "reference":
        reference_unavailable()
        return 0

    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus > 1 and "RANK" not in os.environ:
        # convenience: relaunch under torchrun (the driver already does this itself)
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", str(29500 + os.getpid() % 1000), __file__] + sys.argv[1:]
        return subprocess.call(cmd)

    import torch
    import torch.distributed as dist
    import torch.nn.functional as F
    from torch.nn.parallel import DistributedDataParallel as DDP

    import torch_cgx_b200 as cgx
    from torch_cgx_b200 import models
    from torch_cgx_b200.utils.clocks import ClockSampler
    from torch_cgx_b200.utils.data import CudaPrefetcher, SyntheticHostDataset

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if "MASTER_ADDR" not in os.environ:
        os.environ["MASTER_ADDR"] = "127.0.0.1"
        os.environ["MASTER_PORT"] = str(29400 + os.getpid() % 500)
    dist.init_process_group(args.backend, init_method="env://", rank=rank, world_size=world,
                            device_id=dev if args.backend == "nccl" else None)

    dbatch, dbits, dstoch, unit = MODEL_DEFAULTS[args.model]
    batch = args.batch or dbatch
    bits = dbits if args.bits < 0 else args.bits
    stochastic = dstoch if args.stochastic < 0 else args.stochastic
    if stochastic:
        os.environ["CGX_STOCHASTIC_ROUNDING"] = "1"

    torch.manual_seed(0)
    # same arguments, same results in every run: cuDNN picks convolution algorithms by heuristics,
    # not by timing them (timings vary from process to process), and only deterministic ones
    torch.backends.cudnn.benchmark = False
    torch.backends.cudnn.deterministic = True
    torch.backends.cuda.matmul.allow_tf32 = True
    torch.backends.cudnn.allow_tf32 = True
    is_lm = args.model.startswith("gpt2")
    if args.model == "resnet50":
        net = models.resnet50()
    elif args.model == "resnet18":
        net = models.resnet18()
    elif args.model == "gpt2-medium":
        net = models.gpt2_medium()
    elif args.model == "gpt2-small":
        net = models.gpt2_small()
    elif args.model == "vit-l16":
        net = models.vit_l16()
    else:
        net = models.vit_b16()
    net = net.to(dev)
    if not is_lm:
        net = net.to(memory_format=torch.channels_last)
    nccl_pg = None
    if args.backend == "cgx" and not args.no_nccl_arm:
        nccl_pg = dist.new_group(backend="nccl")  # same-run yardstick: stock NCCL DDP, no hook

    def make_ddp(kind):
        if kind == "nccl_arm":
            return DDP(net, device_ids=[local_rank], gradient_as_bucket_view=True, process_group=nccl_pg)
        d = DDP(net, device_ids=[local_rank], gradient_as_bucket_view=True)
        if args.backend == "cgx":
            state = cgx.CGXState(None, layer_min_size=args.layer_min_size,
                                 compression_params={"bits": bits, "bucket_size": args.bucket_size})
            if args.hook == "native":
                cgx.register_cgx_hook(d, state)
            else:
                d.register_comm_hook(state, cgx.cgx_hook)
        return d

    if is_lm:
        opt = torch.optim.AdamW(net.parameters(), lr=1e-4, fused=True)
    else:
        opt = torch.optim.SGD(net.parameters(), lr=0.05, momentum=0.9, weight_decay=1e-4)

    # synthetic data of the named shape, in PINNED HOST memory (a few distinct batches, cycled)
    if is_lm:
        ds = SyntheticHostDataset.tokens(batch, args.seq_len, net.config.vocab_size, n_batches=4, seed=rank)
        samples_per_step = batch * args.seq_len
    else:
        ds = SyntheticHostDataset.images(batch, 3, 224, 224, 1000, n_batches=4, seed=rank)
        samples_per_step = batch

    ddp = None  # set per arm

    def step(x, y):
        opt.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            if is_lm:
                loss = ddp(x, y)
            else:
                loss = F.cross_entropy(ddp(x), y)
        loss.backward()
        opt.step()
        return loss

    def to_dev(b):
        x, y = b
        x = x.to(dev, non_blocking=True)
        y = y.to(dev, non_blocking=True)
        if not is_lm:
            x = x.contiguous(memory_format=torch.channels_last)
        return x, y

    resident = [to_dev(ds[i]) for i in range(len(ds))]
    torch.cuda.synchronize()
    warm = max(args.warmup, 3)
    native = cgx.get_backend() if args.backend == "cgx" else None
    from torch_cgx_b200.utils.metrics import AsyncScalarReader

    def timed(run_one, k):
        dist.barrier()
        torch.cuda.synchronize()
        if native is not None:
            native.reset_stats()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        last = None
        for i in range(k):
            last = run_one(i)
        e1.record()
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        dist.barrier()
        ms = e0.elapsed_time(e1)
        t = torch.tensor([ms, wall * 1e3], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        launches = native.stats()[1] if native is not None else 0
        return t[0].item(), t[1].item(), launches, last

    def run_arm(capture=None):
        """warm-up + (1) device-timed steps on resident inputs + (2) end-to-end steps (H2D of every
        batch from pinned memory, D2H of every loss) with the CURRENT `ddp`. `capture(loss)` is
        called between (1) and (2), while the model holds what the last step of (1) computed."""
        # W >= 3: DDP rebuilds buckets after step 1, the hook registers layers at step 3
        for i in range(warm):
            step(*resident[i % len(resident)])
        torch.cuda.synchronize()
        ms_dev, _, launches, last_loss = timed(lambda i: step(*resident[i % len(resident)]), args.steps)
        if capture is not None:
            capture(last_loss)
        e2e = None
        if not args.no_e2e:
            pf = CudaPrefetcher(ds, dev, channels_last=not is_lm)
            it = iter(pf)
            for _ in range(2):
                step(*next(it)).item()
            torch.cuda.synchronize()
            reader = AsyncScalarReader(dev, depth=2)

            def one(i):
                x, y = next(it)
                # D2H read of the loss EVERY step (pinned buffer, read one step late so the host
                # keeps enqueueing); the last values are drained inside the timed region below
                reader.push(step(x, y))
                if i == args.steps - 1:
                    reader.drain()
                return None
            _, ms_wall, _, _ = timed(one, args.steps)
            assert len(reader.values) == args.steps, (len(reader.values), args.steps)
            e2e = {"value": round(samples_per_step * world * args.steps / (ms_wall / 1e3), 2), "unit": unit,
                   "h2d_bytes_per_step": ds.bytes_per_batch(), "d2h_bytes_per_step": 4,
                   "ms_per_step": round(ms_wall / args.steps, 3),
                   "timing": "host wall clock around K steps incl. prefetch-stream H2D of every batch and a pinned D2H read of every step's loss (consumed one step late, drained before the clock stops), max over ranks"}
        return ms_dev, launches, last_loss, e2e

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()

    # ---- same-run yardstick: the identical model / step / data on stock NCCL DDP (no compression)
    baseline = None
    if nccl_pg is not None:
        ddp = make_ddp("nccl_arm")
        b_ms, _, _, b_e2e = run_arm()
        baseline = {"what": "same run, same model/step/data: PyTorch DDP over stock NCCL (fp32 gradients, no hook)",
                    "value": round(samples_per_step * world * args.steps / (b_ms / 1e3), 2), "unit": unit,
                    "ms_per_step": round(b_ms / args.steps, 3), "e2e": b_e2e}
        del ddp
        torch.cuda.synchronize()

    # ---- the product arm
    ddp = make_ddp("main")
    outputs = {}
    ms_dev, launches, last_loss, e2e = run_arm(
        capture=(lambda loss: outputs.update(last_step_outputs(net.parameters(), loss)))
        if args.dump_outputs and rank == 0 else None)
    clocks = sampler.stop() if rank == 0 else None

    # ---- allreduce micro-benchmark + correctness self-test at this N (the driver only runs
    # bench.py on several GPUs, so the multi-GPU evidence has to be produced here)
    allreduce_block, selftest_block = None, None
    if args.backend == "cgx" and world > 1:
        if not args.no_selftest:
            import importlib.util

            spec = importlib.util.spec_from_file_location("cgx_selftest", str(ROOT / "bench" / "selftest.py"))
            mod = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(mod)
            selftest_block = mod.run_selftest(dev)
        if not args.no_allreduce:
            allreduce_block = allreduce_microbench(dev, rank, world, nccl_pg, native)

    value = samples_per_step * world * args.steps / (ms_dev / 1e3)
    if rank == 0:
        tag = f"{bits}bit" if args.backend == "cgx" else "nccl_fp32"
        out = {
            "metric": f"{args.model}_ddp_{tag}_{'tokens' if is_lm else 'images'}_per_sec",
            "value": round(value, 2),
            "unit": unit,
            "n_gpus": world,
            "steps": args.steps,
            "warmup": warm,
            "ms_per_step": round(ms_dev / args.steps, 3),
            "higher_is_better": True,
            "scaling": "weak",
            "vs_baseline": round(value / baseline["value"], 4) if baseline else None,
            "baseline": baseline,
            "e2e_vs_baseline": (round(e2e["value"] / baseline["e2e"]["value"], 4)
                                if baseline and e2e and baseline.get("e2e") else None),
            "dtype": "bf16",
            "data": "synthetic (random images/tokens of the named shape, random-init weights)",
            "impl": args.backend,
            "config": {
                "model": args.model, "global_batch": batch * world, "per_gpu_batch": batch,
                "seq_len": args.seq_len if is_lm else None, "image": None if is_lm else 224,
                "parallelism": f"dp{world}", "comm": args.backend, "bits": bits if args.backend == "cgx" else 32,
                "bucket_size": args.bucket_size, "layer_min_size": args.layer_min_size,
                "stochastic_rounding": bool(stochastic), "fusion_buffer_mb": int(os.environ.get("CGX_FUSION_BUFFER_SIZE_MB", "64")),
                "optimizer": "AdamW(fused)" if is_lm else "SGD(momentum)", "grad_dtype": "fp32",
                "l2": "inputs larger than L2: per-step working set (activations+weights+grads) is GBs >> 126 MB L2",
                "lanes": native.lanes() if native is not None else None,
                "hook": args.hook if args.backend == "cgx" else None,
            },
            "gpu_launches": int(launches),
            "e2e": e2e,
            "clocks": clocks,
            "heap": native.heap_kind() if native is not None else None,
            "nvls_multicast": native.uses_multicast() if native is not None else None,
            "allreduce": allreduce_block,
            "selftest": selftest_block,
            "final_loss": round(float(last_loss.detach()), 4) if last_loss is not None else None,
        }
        print(json.dumps(out), flush=True)
        if args.dump_outputs:
            import numpy as np

            out_dir = Path(args.dump_outputs)
            out_dir.mkdir(parents=True, exist_ok=True)
            for name, arr in outputs.items():
                np.save(out_dir / f"{name}.npy", arr)
    dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
