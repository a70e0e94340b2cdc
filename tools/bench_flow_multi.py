"""Data-parallel encode -> decode of the flow graphs (IAN.py / IANv1.py) over N GPUs, one JSON line.

    python -m torch.distributed.run --nproc-per-node N tools/bench_flow_multi.py --graph IAN.py --precision bf16 \
        --per-gpu 512 --gather p2p_async --steps 20 --warmup 5

Every rank holds the same weights (oracle.weights, seed 0) and its own seeded U(-1,1) shard.  --gather picks how the
decoded shards reach every rank:
  p2p_async  the library's pipelined gather: the shard is pushed to the peers on a side stream while the next step
             computes; the last step's gather completes inside the timed region
  p2p        the library's fused gather: the RGB-Beta head's last kernel stores into every rank's buffer + flag barrier
  nccl       ian_reconstruct_dev, then parallel.gather_images (NCCL all_gather)
--per-gpu B is weak scaling (B images per rank); --global-batch G keeps G images over all ranks.  ms_per_step is the
maximum over ranks of CUDA events on the launch stream.  Before timing, one untimed step compares the library's gather
(the fused form when --gather nccl) with parallel.gather_images: gather_check_max_abs_vs_nccl must be 0.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

GFLOP_PER_IMAGE = {"IAN.py": 7.9072}    # SURVEY section 8d; IANv1.py has no committed count


def gpu_info(index):
    """name and power limit of the GPU the numbers were measured on, read in the same run"""
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return {"gpu": out[0], "power_limit_w": float(out[1])}
    except Exception:
        return {"gpu": torch.cuda.get_device_name(index), "power_limit_w": None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--graph", default="IAN.py", choices=["IAN.py", "IANv1.py"])
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--per-gpu", type=int, default=512, help="weak scaling: images per rank")
    ap.add_argument("--global-batch", type=int, default=0, help="same global batch over all ranks (overrides --per-gpu)")
    ap.add_argument("--gather", default="p2p_async", choices=["p2p_async", "p2p", "nccl"])
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 1 or args.per_gpu < 1 or args.global_batch < 0:
        ap.error("--steps, --warmup and --per-gpu must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29561")
    global_n = args.global_batch if args.global_batch else args.per_gpu * world
    if global_n % world:
        raise SystemExit("bench_flow_multi.py: --global-batch must be divisible by the number of ranks")
    n_local = global_n // world
    if not torch.cuda.is_available():
        raise SystemExit("bench_flow_multi.py: no CUDA device")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    import torch.distributed as dist
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)

    from bench import peaks
    from oracle import weights as ow
    pkg = importlib.import_module("neural-photo-editor_b200")
    par = importlib.import_module("neural-photo-editor_b200.parallel")
    W = ow.make_full_weights(0) if args.graph == "IAN.py" else ow.make_v1_weights(0)
    model = pkg.IAN(args.graph, dnn=True, weights=W, device=local_rank)
    model.set_precision(args.precision)
    work = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(work)
    stream = work.cuda_stream

    x = torch.from_numpy(np.random.default_rng(1234 + rank).uniform(-1, 1, (n_local, 3, 64, 64)).astype(np.float32)).to(dev)
    z = torch.empty(n_local, 100, device=dev)
    xhat = torch.empty(n_local, 3, 64, 64, device=dev)

    # one untimed comparison of the library's gather with NCCL's
    model.setup_fused_gather(n_local)
    model.reconstruct_dev(x.data_ptr(), n_local, z.data_ptr(), xhat.data_ptr(), stream)
    want = par.gather_images(xhat, global_n)
    if args.gather == "p2p_async":
        model.reconstruct_gather_async_dev(x.data_ptr(), n_local, z.data_ptr(), stream)
        ptr = model.gather_wait_dev(stream)
    else:
        ptr = model.reconstruct_gather_dev(x.data_ptr(), n_local, z.data_ptr(), stream)
    got = par.as_cuda_tensor(ptr, (global_n, 3, 64, 64), dev)
    check = float((got - want).abs().max().item())
    del want, got

    def step():
        if args.gather == "p2p_async":
            model.reconstruct_gather_async_dev(x.data_ptr(), n_local, z.data_ptr(), stream)
        elif args.gather == "p2p":
            model.reconstruct_gather_dev(x.data_ptr(), n_local, z.data_ptr(), stream)
        else:
            model.reconstruct_dev(x.data_ptr(), n_local, z.data_ptr(), xhat.data_ptr(), stream)
            par.gather_images(xhat, global_n)

    def finish():
        if args.gather == "p2p_async":
            model.gather_wait_dev(stream)                   # the last step's gather lands inside the timed region

    for _ in range(args.warmup):
        step()
    finish()
    dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step()
    finish()
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1), check], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, check = float(t[0]) / args.steps, float(t[1])
    info = gpu_info(local_rank)

    if rank == 0:
        ips = global_n / (ms / 1e3)
        line = {"metric": "64x64 images/sec %s encode->decode, %d GPUs, all-gather of the decoded images" % (args.graph, world),
                "value": ips, "unit": "images/sec", "graph": args.graph, "precision": args.precision, "n_gpus": world,
                "per_gpu": n_local, "global_batch": global_n, "scaling": "strong" if args.global_batch else "weak",
                "gather": args.gather, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
                "gather_check_max_abs_vs_nccl": check, "gather_check_form": "p2p" if args.gather == "nccl" else args.gather,
                **info}
        if args.graph in GFLOP_PER_IMAGE:
            pk = peaks()
            peak = pk["bf16_tflops"] / (1.0 if args.precision == "bf16" else 3.0)   # fp32: 3 bf16 passes, as in bench.py
            line["tflops_algorithmic"] = ips * GFLOP_PER_IMAGE[args.graph] / 1e3
            line["whole_step_frac_burst"] = line["tflops_algorithmic"] / world / peak
            line["peak_note"] = "per GPU, %s bf16_tflops %.1f (burst)%s" % (pk["src"], pk["bf16_tflops"],
                                                                            "" if args.precision == "bf16" else " / 3")
        print(json.dumps(line), flush=True)
    model.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
