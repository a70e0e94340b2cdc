"""bench.py -- BASELINE metric: 64x64 images/sec, IAN_simple encode -> decode @ batch 256 (fp32 semantics),
plus latent-edit steps/sec as a secondary block.  Contract: see the task statement / DESIGN.md section 5.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--global-batch G] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

`--dump-outputs DIR` (one GPU) writes what the last timed step returned -- the latents z and the decoded images xhat -- as
DIR/z.npy and DIR/xhat.npy (float32).  Inputs and weights are seeded, so two builds can be compared output for output.

Default: weak scaling, 256 images per GPU (BASELINE configs[1] on every GPU).  `--global-batch G` shards a FIXED global
batch (BASELINE configs[4]: 4096) over the ranks (strong scaling); the default run also reports that configuration as
the secondary block `config5`, so the driver's 1/2/4/8-GPU runs carry the same-global-batch curve.
"""
from __future__ import annotations

import argparse
import atexit
import importlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BATCH = 256                      # per-GPU batch (BASELINE configs[1]); weak scaling over GPUs
EDIT_BATCH, EDIT_STEPS = 128, 32  # BASELINE configs[3]
GFLOP_PER_IMAGE = 2.5921488      # SURVEY Appendix E: 1 296 074 400 MAC, encode -> decode
# MACs per image executed by the tap-GEMM kernel (enc_conv2-4, enc_fc1, heads, l_dec_fc2, dec_conv1-3)
TAPGEMM_LAYERS = {"enc_conv2": 209715200, "enc_conv3": 209715200, "enc_conv4": 209715200, "enc_fc1": 16384000,
                  "enc_head": 200000, "l_dec_fc2": 1638400, "dec_conv1": 209715200, "dec_conv2": 209715200,
                  "dec_conv3": 209715200}
EDGE_KERNELS = ("enc_conv1", "dec_out")
# algorithmic HBM bytes per image of the two HBM-bound end kernels: x in + a1 planes out / h3 planes in + x_hat out
EDGE_BYTES_PER_IMAGE = {"enc_conv1": 49152 + 32 * 32 * 128 * 4, "dec_out": 32 * 32 * 128 * 4 + 49152}
CONFIG5_GLOBAL = 4096            # BASELINE configs[4]
NCU_SUMMARY = os.path.join(ROOT, "profiles", "r2_ncu_tc_kernels_full_summary.csv")
METRIC = "64x64 images/sec IAN encode->decode @ batch 256"
DUMP_MAX_ROWS = 1024             # --dump-outputs: 1024 decoded images are 50 MB of float32, under the 64 MB a dump may take


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "src": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "src": "fallback"}


def ncu_traffic(kernel_substr, launches_per_step):
    """dram__bytes_read + dram__bytes_write of the first `launches_per_step` launches whose kernel name contains
    `kernel_substr`, from the committed `ncu --set full` summary of this same command (tools/ncu_summary.py); None if the
    file is absent.  Not a measurement of the run that prints it -- the file it came from is named beside it."""
    import csv
    if not os.path.exists(NCU_SUMMARY):
        return None
    rows = list(csv.reader(open(NCU_SUMMARY)))
    hdr = rows[0]
    try:
        kn = [i for i, h in enumerate(hdr) if h.startswith("Kernel Name")][0]
        rd = [i for i, h in enumerate(hdr) if h.startswith("dram__bytes_read.sum")][0]
        wr = [i for i, h in enumerate(hdr) if h.startswith("dram__bytes_write.sum")][0]
    except IndexError:
        return None
    scale = {"Mbyte": 1e6, "Gbyte": 1e9, "Kbyte": 1e3, "byte": 1.0}
    unit_r = hdr[rd].split("[")[-1].rstrip("]")
    unit_w = hdr[wr].split("[")[-1].rstrip("]")
    tot, n = 0.0, 0
    for r in rows[1:]:
        if kernel_substr in r[kn] and n < launches_per_step:
            tot += float(r[rd]) * scale.get(unit_r, 1.0) + float(r[wr]) * scale.get(unit_w, 1.0)
            n += 1
    return tot if n == launches_per_step else None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe): one
    background `nvidia-smi -lms 20` process; samples are selected by wall-clock window."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        fd, self.path = tempfile.mkstemp(prefix="ian_clocks_%d_" % index, suffix=".csv")
        self.f = os.fdopen(fd, "w")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"], stdout=self.f,
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None
        atexit.register(self._end)                          # the sampler never outlives the run, however it ends
        self.t0 = self.t1 = None

    def _end(self):
        if self.proc is not None and self.proc.poll() is None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
        self.f.close()

    def start(self):
        self.t0 = time.time()

    def stop(self):
        self.t1 = time.time()

    def summary(self):
        import datetime
        if self.proc is not None:
            time.sleep(0.05)
        self._end()
        rows_all, rows_in = [], []
        for line in open(self.path):
            c = [v.strip() for v in line.split(",")]
            if len(c) < 8:
                continue
            try:
                ts = datetime.datetime.strptime(c[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                sm, mx, pw = float(c[1]), float(c[2]), float(c[3])
            except Exception:
                continue
            row = (sm, mx, pw, c[4:8])
            rows_all.append(row)
            if self.t0 is not None and self.t0 - 0.01 <= ts <= (self.t1 or 1e18) + 0.01:
                rows_in.append(row)
        try:
            os.remove(self.path)
        except OSError:
            pass
        rows = rows_in if rows_in else rows_all
        reasons = set()
        for r in rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median([r[0] for r in rows])) if rows else None,
                "sm_max_mhz": max(r[1] for r in rows) if rows else None,
                "power_w_max": max(r[2] for r in rows) if rows else None,
                "reasons": sorted(reasons), "samples": len(rows),
                "window": "timed region" if rows_in else "whole run (timed region shorter than the sampling period)"}


def _cpu_setup():
    from oracle import ian_torch as ot
    from oracle import weights as ow
    P = ot.to_torch(ow.make_simple_weights(0), torch.float32)
    return ot, P


def _pick_threads(ot, P, x):
    """torch oversubscribes badly when the container is cpu-limited: time one batch per candidate thread count."""
    try:
        avail = len(os.sched_getaffinity(0))
    except Exception:
        avail = os.cpu_count() or 1
    best, best_t = 1, float("inf")
    for th in sorted({avail, 64, 32, 16, 8}, reverse=True):
        if th > avail:
            continue
        torch.set_num_threads(th)
        with torch.no_grad():
            ot.decode(P, ot.encode(P, x))
            t0 = time.perf_counter()
            ot.decode(P, ot.encode(P, x))
            dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = th, dt
    torch.set_num_threads(best)
    return best, avail


def cpu_restatement_rate(seconds_budget=12.0, batch=32):
    """The reference's Theano CPU path cannot run (SURVEY F3): time the float32 torch restatement of the
    reference graph on the host cores, on a bounded sample of the same workload."""
    ot, P = _cpu_setup()
    x = torch.from_numpy(np.random.default_rng(1234).uniform(-1, 1, (batch, 3, 64, 64)).astype(np.float32))
    threads, avail = _pick_threads(ot, P, x)
    with torch.no_grad():
        t0, n = time.perf_counter(), 0
        while True:
            ot.decode(P, ot.encode(P, x))
            n += 1
            if time.perf_counter() - t0 > seconds_budget or n >= 64:
                break
        dt = time.perf_counter() - t0
    return {"value": batch * n / dt, "unit": "images/sec", "cores": threads, "kind": "port",
            "sample": "%d x batch-%d encode->decode of the float32 torch-CPU restatement (oracle/ian_torch.py), %.1f s; "
                      "%d threads picked by calibration out of %d available" % (n, batch, dt, threads, avail)}


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path = CPU restatement (port)."""
    if rank != 0:
        return
    t_all = time.perf_counter()
    ot, P = _cpu_setup()
    sample = BATCH                                          # every step is the real batch-256 workload (about 1 s of CPU)
    x = torch.from_numpy(np.random.default_rng(1234).uniform(-1, 1, (sample, 3, 64, 64)).astype(np.float32))
    threads, avail = _pick_threads(ot, P, x[:32])
    with torch.no_grad():
        for _ in range(args.warmup):
            ot.decode(P, ot.encode(P, x))
        t0 = time.perf_counter()
        for _ in range(args.steps):
            ot.decode(P, ot.encode(P, x))
        dt = time.perf_counter() - t0
    v = sample * args.steps / dt
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "images/sec", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "IAN_simple encode->decode, batch 256 per GPU (BASELINE configs[1])",
                       "global_batch": BATCH * world,
                       "note": "reference Theano path cannot run here (py2/theano absent); this is the CPU restatement "
                               "of the reference graph on %d host threads (of %d available), each step one batch of %d images"
                               % (threads, avail, sample)},
            "cpu_baseline": {"value": v, "unit": "images/sec", "cores": threads, "kind": "port",
                             "sample": "%d steps x %d images" % (args.steps, sample)},
            "e2e": {"value": v, "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "wall_s": time.perf_counter() - t_all}
    print(json.dumps(line), flush=True)


def _psnr(a, b):
    """PSNR (dB) on the [-1,1] image range (peak-to-peak 2)."""
    mse = float(((a - b) ** 2).mean().item())
    return float("inf") if mse == 0 else 10.0 * float(np.log10(4.0 / mse))


def dump_outputs(out_dir, arrays):
    """--dump-outputs: each CUDA tensor as out_dir/<name>.npy in float32.  An array of more than DUMP_MAX_ROWS rows keeps
    the rows of a fixed seeded sample (ascending), so the dumps of two builds hold the same rows."""
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        a = t.float().cpu().numpy()
        if a.shape[0] > DUMP_MAX_ROWS:
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], DUMP_MAX_ROWS, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--global-batch", type=int, default=0,
                    help="0 (default): weak scaling, 256 images per GPU.  G > 0: strong scaling, G images sharded over the ranks")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-edit", action="store_true")
    ap.add_argument("--no-full", action="store_true", help="skip the full-IAN (BASELINE configs[2]) block")
    ap.add_argument("--no-config5", action="store_true", help="skip the global-batch-4096 block (BASELINE configs[4])")
    ap.add_argument("--gather", default="p2p_async", choices=["p2p_async", "p2p", "nccl"],
                    help="N>1: p2p_async = decoded shard pushed to the peers on a side stream (copy engines + stream memory "
                         "operations; IAN_PUSH=kernel: a copy kernel) while the next step computes (default); p2p = peer stores fused into the dec_out kernel; nccl = separate NCCL all_gather")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write z and xhat of the last timed step as DIR/z.npy and DIR/xhat.npy (float32; one GPU)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.dump_outputs and (world > 1 or args.impl != "ours"):
        ap.error("--dump-outputs dumps the CUDA path on one GPU")
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the IAN hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    from oracle import weights as ow                        # weight / input GENERATORS only (synthetic checkpoint)
    pkg = importlib.import_module("neural-photo-editor_b200")
    par = importlib.import_module("neural-photo-editor_b200.parallel")
    W_simple = ow.make_simple_weights(0)
    dev = torch.device("cuda", local_rank)
    work_stream = torch.cuda.Stream(device=dev)             # non-default stream: its handle is what the C-ABI takes
    torch.cuda.set_stream(work_stream)
    stream = work_stream.cuda_stream
    assert stream != 0

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(*vals):
        if world == 1:
            return [float(v) for v in vals]
        t = torch.tensor(list(vals), device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t.tolist()]

    def timed_job(model, n_local, global_n, seed, steps, warmup, gather_mode, sampler=None, dump_dir=None):
        """K steps of encode -> decode of this rank's shard (+ the all-gather of the decoded images at N>1), device timed.
        Returns (ms_total max over ranks, launches, gather_check, gather_mode actually used).  With `dump_dir` (one GPU),
        the last timed step's z and xhat are written there once the timed region has ended."""
        rng = np.random.default_rng(seed + rank)
        x = torch.from_numpy(rng.uniform(-1, 1, (n_local, 3, 64, 64)).astype(np.float32)).to(dev)
        z = torch.empty(n_local, 100, device=dev)
        xhat = torch.empty(n_local, 3, 64, 64, device=dev)
        check = None
        if world > 1 and gather_mode != "nccl":
            try:
                model.setup_fused_gather(n_local)
                # one untimed cross-check of the library's gather against NCCL's all_gather (parallel.gather_images)
                model.reconstruct_dev(x.data_ptr(), n_local, z.data_ptr(), xhat.data_ptr(), stream)
                want = par.gather_images(xhat, global_n)
                if gather_mode == "p2p":
                    ptr = model.reconstruct_gather_dev(x.data_ptr(), n_local, z.data_ptr(), stream)
                else:
                    model.reconstruct_gather_async_dev(x.data_ptr(), n_local, z.data_ptr(), stream)
                    ptr = model.gather_wait_dev(stream)
                got = par.as_cuda_tensor(ptr, (global_n, 3, 64, 64), dev)
                check = float((got - want).abs().max().item())
                del want
            except Exception as e:                          # e.g. CUDA IPC not permitted in this container
                gather_mode = "nccl"
                check = "p2p setup failed: %s" % (str(e)[:120],)

        def step():
            if world > 1 and gather_mode == "p2p_async":
                model.reconstruct_gather_async_dev(x.data_ptr(), n_local, z.data_ptr(), stream)
            elif world > 1 and gather_mode == "p2p":
                model.reconstruct_gather_dev(x.data_ptr(), n_local, z.data_ptr(), stream)
            else:
                model.reconstruct_dev(x.data_ptr(), n_local, z.data_ptr(), xhat.data_ptr(), stream)
                if world > 1:
                    par.gather_images(xhat, global_n)       # the one collective of the path (north_star), via NCCL

        def finish():
            if world > 1 and gather_mode == "p2p_async":
                model.gather_wait_dev(stream)               # the last step's gather must land inside the timed region

        for _ in range(warmup):
            step()
        finish()
        barrier()
        if sampler is not None:
            sampler.start()                                 # nvidia-smi clock samples are selected by this window
        l0 = model.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step()
        finish()
        e1.record()
        barrier()
        if sampler is not None:
            sampler.stop()
        launches = model.launch_count() - l0
        if dump_dir is not None:
            dump_outputs(dump_dir, {"z": z, "xhat": xhat})
        (ms,) = max_over_ranks(e0.elapsed_time(e1))
        return ms, launches, check, gather_mode, step, x

    strong = args.global_batch > 0
    global_n = args.global_batch if strong else BATCH * world
    if global_n % world:
        raise SystemExit("bench.py: --global-batch must be divisible by the number of ranks")
    lo, hi = par.shard_bounds(global_n, rank, world)
    n_local = hi - lo
    model = pkg.IAN("IAN_simple.py", dnn=True, weights=W_simple, device=local_rank)
    torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    ms, launches, gather_check, gather_mode, step, x = timed_job(model, n_local, global_n, 1234, args.steps, args.warmup,
                                                                 args.gather if world > 1 else "none", sampler,
                                                                 args.dump_outputs)
    value = global_n * args.steps / (ms / 1e3)

    # ---- roofline of the dominant kernel (tap-GEMM), CUDA events on the launch stream, same loop
    model.set_layer_timing(True)
    for _ in range(max(3, args.steps // 3)):
        step()
    torch.cuda.synchronize()
    model.set_layer_timing(False)
    layer_ms = {k: model.layer_time_ms(k) for k in TAPGEMM_LAYERS}
    edge_ms = {k: model.layer_time_ms(k) for k in EDGE_KERNELS}
    chunks = (n_local + 511) // 512                         # layer times are per launch; a step of > 512 images is `chunks` launches
    tg_ms = sum(v for v in layer_ms.values() if v > 0) * chunks
    per_launch_imgs = n_local / chunks
    tg_flops = 2.0 * sum(TAPGEMM_LAYERS.values()) * n_local
    pk = peaks()
    achieved = tg_flops / (tg_ms / 1e3) / 1e12 if tg_ms > 0 else 0.0
    peak_burst, peak_sust = pk["bf16_tflops"] / 3.0, pk["bf16_tflops_sustained"] / 3.0
    timed_region_ms = ms
    traffic = ncu_traffic("tapgemm_tc", len(TAPGEMM_LAYERS)) if (n_local == BATCH and world == 1) else None
    hbm = pk["hbm_gbs"]
    edge_roof = {k: {"ms": round(edge_ms[k], 4), "algorithmic_mb": round(EDGE_BYTES_PER_IMAGE[k] * per_launch_imgs / 1e6, 1),
                     "achieved_gbs": round(EDGE_BYTES_PER_IMAGE[k] * per_launch_imgs / (edge_ms[k] / 1e3) / 1e9, 1),
                     "frac_of_measured_hbm": round(EDGE_BYTES_PER_IMAGE[k] * per_launch_imgs / (edge_ms[k] / 1e3) / 1e9 / hbm, 3)}
                 for k in EDGE_KERNELS if edge_ms[k] > 0}
    roofline = {"bound": "tensor", "kernel": "tapgemm_tc_kernel", "achieved": achieved, "unit": "TFLOP/s",
                # the timed region is a few tens of ms at full clocks: the BURST figure is the honest denominator; the
                # sustained one (seconds-long cuBLAS loop under the power cap) is printed beside it
                "peak": peak_burst, "frac": achieved / peak_burst,
                "frac_burst": achieved / peak_burst, "frac_sustained": achieved / peak_sust,
                "peak_burst": peak_burst, "peak_sustained": peak_sust, "timed_region_ms": timed_region_ms,
                "peak_note": "%s bf16_tflops %.1f (burst) / %.1f (sustained), each / 3: float32 parity is reached by a 3-pass "
                             "bf16 split, so one algorithmic MAC costs 3 tensor-core MACs" % (pk["src"], pk["bf16_tflops"], pk["bf16_tflops_sustained"]),
                "tensor_executed_tflops": 3 * achieved, "kernel_ms_per_step": tg_ms,
                "algorithmic_flop_per_step": tg_flops,
                "traffic": traffic, "traffic_unit": "bytes per step, dram read+write summed over the 9 tap-GEMM launches",
                "traffic_src": os.path.relpath(NCU_SUMMARY, ROOT) if traffic is not None else None,
                "traffic_algorithmic": 943.0e6 if n_local == BATCH else None,
                # share among the kernels event-timed in this same pass (tap-GEMMs + enc_conv1 + dec_out)
                "kernel_share_of_step": tg_ms / (tg_ms + chunks * sum(v for v in edge_ms.values() if v > 0)),
                "kernel_ms_vs_untimed_step": tg_ms / (ms / args.steps),
                "whole_step_frac_burst": (value / world) * GFLOP_PER_IMAGE / 1e3 / peak_burst,
                "layer_ms": {k: round(v, 4) for k, v in layer_ms.items()},
                "edge_kernel_ms": {k: round(v, 4) for k, v in edge_ms.items()},
                "edge_kernels_hbm": edge_roof}

    # ---- e2e through the public API with HOST buffers (H2D + D2H of every step inside the timed region).
    # (a) the streaming call IAN.reconstruct_stream (two batches in flight, pinned buffers) -> e2e.value;
    # (b) the synchronous call IAN.reconstruct(x, out=pinned); (c) the plain drop-in call IAN.reconstruct(x) on
    # pageable numpy arrays with a fresh pageable result per call.
    EB = min(n_local, 512)
    x_host = torch.from_numpy(np.random.default_rng(1234 + rank).uniform(-1, 1, (EB, 3, 64, 64)).astype(np.float32)).pin_memory()
    x_np = x_host.numpy()
    x_pageable = x_np.copy()
    out_pinned = model.pinned_empty((EB, 3, 64, 64))
    for _ in range(3):
        model.reconstruct(x_np, out=out_pinned)
        model.reconstruct(x_pageable)
    barrier()
    e2e_steps = max(5, args.steps)
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        model.reconstruct(x_np, out=out_pinned)
    t_sync = time.perf_counter() - t0
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        model.reconstruct(x_pageable)
    t_page = time.perf_counter() - t0
    for _ in model.reconstruct_stream(x_np for _ in range(3)):
        pass
    barrier()
    t0 = time.perf_counter()
    checksum = 0.0
    for xh in model.reconstruct_stream(x_np for _ in range(e2e_steps)):
        checksum += float(xh[0, 0, 0, 0])                   # touch every result on the host
    t_pipe = time.perf_counter() - t0
    t_sync, t_pipe, t_page = max_over_ranks(t_sync, t_pipe, t_page)
    e2e = {"value": world * EB * e2e_steps / t_pipe, "unit": "images/sec", "h2d_bytes_per_step": EB * 12288 * 4,
           "d2h_bytes_per_step": EB * 12288 * 4,
           "api": "IAN.reconstruct_stream(batches of numpy (%d,3,64,64) in pinned memory): 2 batches in flight, "
                  "every batch is copied H2D, encoded, decoded and copied D2H" % EB,
           "sync_value": world * EB * e2e_steps / t_sync,
           "sync_api": "IAN.reconstruct(x, out=pinned) -> ian_reconstruct_host, one batch at a time",
           "pageable_value": world * EB * e2e_steps / t_page,
           "pageable_api": "IAN.reconstruct(x): pageable numpy in, fresh pageable numpy out -- the plain drop-in call",
           "steps": e2e_steps,
           "note": None if world == 1 else "e2e at N>1 = N independent host streams (each rank copies its own batches in "
                                           "and out); no all-gather is part of it, unlike `value`"}

    # ---- BASELINE configs[4]: global batch 4096 sharded over the ranks (same global batch at every N)
    config5 = None
    if not args.no_config5 and not strong and CONFIG5_GLOBAL % world == 0:
        m5 = pkg.IAN("IAN_simple.py", dnn=True, weights=W_simple, device=local_rank) if world > 1 else model
        l5, h5 = par.shard_bounds(CONFIG5_GLOBAL, rank, world)
        s5 = max(3, args.steps // 4)
        ms5, _, chk5, mode5, _, _ = timed_job(m5, h5 - l5, CONFIG5_GLOBAL, 4321, s5, 3, args.gather if world > 1 else "none")
        config5 = {"metric": "64x64 images/sec IAN_simple encode->decode, global batch 4096 sharded over %d GPU(s) "
                             "(BASELINE configs[4])" % world, "value": CONFIG5_GLOBAL * s5 / (ms5 / 1e3), "unit": "images/sec",
                   "scaling": "strong", "global_batch": CONFIG5_GLOBAL, "per_gpu": h5 - l5, "steps": s5,
                   "ms_per_step": ms5 / s5, "gather": mode5, "gather_check_max_abs_vs_nccl": chk5,
                   "frac_burst_whole_step": CONFIG5_GLOBAL * s5 / (ms5 / 1e3) / world * GFLOP_PER_IMAGE / 1e3 / peak_burst}
        if m5 is not model:
            m5.close()

    # ---- secondary metric: latent-edit steps/sec (BASELINE configs[3])
    edit = None
    if not args.no_edit and world == 1:                      # secondary blocks are single-GPU measurements
        z_np, boxes_np, rgb_np = ow.config4_inputs(EDIT_BATCH)   # SURVEY 8d config 4: seeds 2/3, NPE's box law
        ze, boxes, rgb = (torch.from_numpy(a).to(dev) for a in (z_np, boxes_np, rgb_np))
        # one whole 32-step loop as warm-up, then EDIT_REPS timed loops back to back (each from the same start latents,
        # events around each loop); the MEDIAN loop is reported -- a single 27 ms loop after an idle gap measured the
        # clock ramp as much as the kernels (+-15 % between runs of one build on one box)
        zw = ze.clone()
        model.edit_loop_dev(zw.data_ptr(), boxes.data_ptr(), rgb.data_ptr(), 0, EDIT_BATCH, EDIT_STEPS, 0.05, stream)
        EDIT_REPS = 5
        zws = [ze.clone() for _ in range(EDIT_REPS)]
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(EDIT_REPS)]
        torch.cuda.synchronize()
        for zr, (a0, a1) in zip(zws, evs):
            a0.record()
            model.edit_loop_dev(zr.data_ptr(), boxes.data_ptr(), rgb.data_ptr(), 0, EDIT_BATCH, EDIT_STEPS, 0.05, stream)
            a1.record()
        torch.cuda.synchronize()
        loops_ms = sorted(a0.elapsed_time(a1) for a0, a1 in evs)
        ems = loops_ms[EDIT_REPS // 2]
        etf = 2.5625 * EDIT_BATCH * EDIT_STEPS / (ems / 1e3) / 1e3
        edit = {"metric": "latent-edit steps/sec (32-step dL/dz descent, batch 128)", "value": EDIT_STEPS * EDIT_BATCH / (ems / 1e3),
                "unit": "sample-steps/sec", "loop_iters_per_sec": EDIT_STEPS / (ems / 1e3), "ms_total": ems,
                "ms_total_min_max": [loops_ms[0], loops_ms[-1]], "loops_timed": EDIT_REPS,
                "tflops": etf, "frac_burst": etf / peak_burst}

    # ---- BASELINE configs[0] size: one image, encode -> decode, through the synchronous host API (NPE's call pattern)
    lat = None
    if rank == 0 and world == 1:
        x1 = x_np[:1].copy()
        for _ in range(5):
            model.reconstruct(x1)
        ts = []
        for _ in range(30):
            t0 = time.perf_counter()
            model.reconstruct(x1)
            ts.append(time.perf_counter() - t0)
        lat = {"batch": 1, "median_ms": 1e3 * float(np.median(ts)), "min_ms": 1e3 * float(np.min(ts)),
               "api": "IAN.reconstruct(numpy (1,3,64,64)), synchronous, includes H2D/D2H"}
        # one NPE paint stroke (NPE.py:199-231): gradient step on Z, re-decode, DELTA/MASK/ERROR blend, 256x256 display
        z1 = model.encode_images(x1)
        recon = np.uint8((model.sample_at(z1)[0] + 1.0) * 127.5)
        err = np.zeros((3, 64, 64), np.float32)
        frame = np.full((1, 3, 64, 64), 0.25, np.float32)
        box = [20.0, 20.0, 30.0, 30.0]
        for _ in range(5):
            model.paint_stroke(z1, box, frame, recon, err)
        ts = []
        for _ in range(30):
            t0 = time.perf_counter()
            model.paint_stroke(z1, box, frame, recon, err)
            ts.append(time.perf_counter() - t0)
        lat["paint_stroke_median_ms"] = 1e3 * float(np.median(ts))
        lat["paint_stroke_api"] = "IAN.paint_stroke: one library call per stroke, kernels replayed as one CUDA graph"

    # ---- secondary block: full IAN (reference IAN.py graph), BASELINE configs[2] size (batch 512)
    full = None
    if not args.no_full and rank == 0 and world == 1:
        fm = pkg.IAN("IAN.py", dnn=True, weights=ow.make_full_weights(0), device=local_rank)
        FB = 512
        xf = torch.from_numpy(np.random.default_rng(77).uniform(-1, 1, (FB, 3, 64, 64)).astype(np.float32)).to(dev)
        zf = torch.empty(FB, 100, device=dev)
        xhf = torch.empty(FB, 3, 64, 64, device=dev)
        names = ["enc_conv1", "enc_conv2", "enc_conv3", "enc_conv4", "enc_fc1", "enc_head", "full_dec_fc2", "full_dec_conv1", "dec_conv2a",
                 "dec_conv2a2", "full_dec_conv2", "dec_conv3a", "dec_conv3a2", "full_dec_conv3", "dec_conv4a", "dec_conv4a2",
                 "full_dec_conv4", "rgb_head"]
        fsteps = max(3, args.steps // 6)
        res, outs = {}, {}
        for prec in ("fp32", "bf16"):
            fm.set_precision(prec)
            torch.cuda.synchronize()
            for _ in range(3):
                fm.reconstruct_dev(xf.data_ptr(), FB, zf.data_ptr(), xhf.data_ptr(), stream)
            torch.cuda.synchronize()
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record()
            for _ in range(fsteps):
                fm.reconstruct_dev(xf.data_ptr(), FB, zf.data_ptr(), xhf.data_ptr(), stream)
            f1.record()
            torch.cuda.synchronize()
            fms = f0.elapsed_time(f1) / fsteps
            fm.set_layer_timing(True)
            fm.reconstruct_dev(xf.data_ptr(), FB, zf.data_ptr(), xhf.data_ptr(), stream)
            torch.cuda.synchronize()
            fm.set_layer_timing(False)
            outs[prec] = xhf.clone()
            tfa = 7.9072 * FB / (fms / 1e3) / 1e3
            res[prec] = {"value": FB / (fms / 1e3), "ms_per_step": fms, "tflops_algorithmic": tfa,
                         "frac_burst": tfa / (pk["bf16_tflops"] / (1.0 if prec == "bf16" else 3.0)),
                         "layer_ms": {k: round(fm.layer_time_ms(k), 4) for k in names}}
        diff = (outs["bf16"] - outs["fp32"]).abs()
        full = {"metric": "64x64 images/sec full IAN (IAN.py) encode->decode @ batch 512 (BASELINE configs[2])",
                "unit": "images/sec", "value": res["bf16"]["value"], "dtype": "bf16 operands, fp32 accumulate (single tcgen05 pass)",
                "bf16": res["bf16"], "fp32_split": res["fp32"],
                "bf16_vs_fp32_max_abs": float(diff.max().item()), "bf16_vs_fp32_mean_abs": float(diff.mean().item()),
                "bf16_vs_fp32_psnr_db": _psnr(outs["bf16"], outs["fp32"])}
        fm.close()

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_restatement_rate()

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "images/sec", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
                "scaling": "strong" if strong else "weak",
                "vs_baseline": None, "dtype": "f32 (3-pass bf16 split on tcgen05, fp32 accumulate)", "data": "synthetic",
                "config": {"workload": ("IAN_simple encode->decode, global batch %d sharded over the ranks (BASELINE configs[4])" % global_n)
                           if strong else "IAN_simple encode->decode, batch 256 per GPU (BASELINE configs[1])",
                           "global_batch": global_n, "per_gpu": n_local, "parallelism": "dp%d" % world,
                           "l2": "no flush: one step streams 211 MB of weights + ~1 GB of activations (> 126 MB L2)",
                           "collective": {"none": "none", "nccl": "NCCL all_gather of decoded images after dec_out",
                                          "p2p": "all-gather fused into dec_out: st.global to every rank's buffer over NVLink "
                                                 "peer memory + flag barrier",
                                          "p2p_async": "all-gather by the library's own side-stream push over NVLink peer memory (copy engines + "
                                                       "stream memory operations unless IAN_PUSH=kernel; free/pushed flag handshake), overlapped with the next step's tensor kernels; "
                                                       "the last step's gather completes inside the timed region"}[gather_mode],
                           "gather_check_max_abs_vs_nccl": gather_check},
                "tflops_algorithmic": value * GFLOP_PER_IMAGE / 1e3, "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e,
                "gpu_launches": launches, "clocks": sampler.summary(), "config5": config5, "edit": edit, "full_ian": full,
                "single_image_latency": lat}
        print(json.dumps(line), flush=True)
    model.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
