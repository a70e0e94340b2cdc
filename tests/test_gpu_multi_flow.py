"""The library's all-gather on the flow graphs (IAN.py, IANv1.py): the RGB-Beta head's last kernel stores the decoded
images into every rank's gather buffer, as dec_out does for IAN_simple (tests/test_gpu_multi.py).

The gathered images must equal, bit for bit, what ian_reconstruct_dev returns for the same shard at the same batch size:
the same kernels run with the same schedule, and the header promises the same bits for a repeated call.

  * one GPU: a single-process NCCL group of world 1, every (graph, precision, gather form), three steps per case so both
    gather-buffer halves are used; the verification path refuses the gather calls
  * two GPUs: two spawned processes with rank skew, small-batch (split-K) and CTA-pair shard sizes, and
    IAN.reconstruct_sharded with a shard above the 512-image plan chunk.  Skipped with fewer than 2 GPUs.
"""
import importlib
import os
import socket
import sys
import traceback

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GRAPHS = ("IAN.py", "IANv1.py")


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _weights(graph):
    from oracle import weights as ow
    return ow.make_full_weights(0) if graph == "IAN.py" else ow.make_v1_weights(0)


def _images(seed, n, dev):
    import torch
    return torch.from_numpy(np.random.default_rng(seed).uniform(-1, 1, (n, 3, 64, 64)).astype(np.float32)).to(dev)


# ---- one GPU --------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def world1():
    import torch.distributed as dist
    saved = {k: os.environ.get(k) for k in ("MASTER_ADDR", "MASTER_PORT")}
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(_free_port())
    dist.init_process_group("nccl", rank=0, world_size=1)
    yield
    dist.destroy_process_group()
    for k, v in saved.items():
        if v is None:
            os.environ.pop(k, None)
        else:
            os.environ[k] = v


N_LOCAL_1 = 6


@pytest.fixture(scope="module", params=GRAPHS)
def flow_model(request, npe, world1):
    """one handle per graph: gather buffers cannot be re-created on a handle, precision is switched on the live one"""
    m = npe.IAN(request.param, dnn=True, weights=_weights(request.param), device=0)
    m.setup_fused_gather(N_LOCAL_1)
    yield m
    m.close()


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("pipelined", [False, True], ids=["fused", "pipelined"])
def test_flow_gather_world1_is_bit_identical_to_reconstruct_dev(flow_model, precision, pipelined):
    import torch
    par = importlib.import_module("neural-photo-editor_b200.parallel")
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(device=dev)
    flow_model.set_precision(precision)
    n = N_LOCAL_1
    try:
        with torch.cuda.stream(stream):
            for t in range(3):                                  # alternating gather-buffer halves
                x = _images(40 + t, n, dev)
                want, z_want = torch.empty_like(x), torch.empty(n, 100, device=dev)
                z_got = torch.full((n, 100), float("nan"), device=dev)
                flow_model.reconstruct_dev(x.data_ptr(), n, z_want.data_ptr(), want.data_ptr(), stream.cuda_stream)
                if pipelined:
                    flow_model.reconstruct_gather_async_dev(x.data_ptr(), n, z_got.data_ptr(), stream.cuda_stream)
                    ptr = flow_model.gather_wait_dev(stream.cuda_stream)
                else:
                    ptr = flow_model.reconstruct_gather_dev(x.data_ptr(), n, z_got.data_ptr(), stream.cuda_stream)
                got = par.as_cuda_tensor(ptr, (n, 3, 64, 64), dev).clone()
                stream.synchronize()
                assert torch.equal(got, want), (t, float((got - want).abs().max()))
                assert torch.equal(z_got, z_want), (t, float((z_got - z_want).abs().max()))
    finally:
        flow_model.set_precision("fp32")


def test_flow_gather_refused_on_the_verification_path(flow_model, npe):
    import torch
    x = _images(3, N_LOCAL_1, torch.device("cuda", 0))
    flow_model.set_path("simt")
    try:
        with pytest.raises(npe.IanError):
            flow_model.reconstruct_gather_dev(x.data_ptr(), N_LOCAL_1)
        with pytest.raises(npe.IanError):
            flow_model.reconstruct_gather_async_dev(x.data_ptr(), N_LOCAL_1)
    finally:
        flow_model.set_path("tc")


# ---- two GPUs -------------------------------------------------------------------------------------------------------
def _worker(rank, world, port, q):
    try:
        if ROOT not in sys.path:
            sys.path.insert(0, ROOT)
        import torch
        import torch.distributed as dist
        os.environ["MASTER_ADDR"] = "127.0.0.1"
        os.environ["MASTER_PORT"] = str(port)
        torch.cuda.set_device(rank)
        dev = torch.device("cuda", rank)
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
        pkg = importlib.import_module("neural-photo-editor_b200")
        par = importlib.import_module("neural-photo-editor_b200.parallel")
        stream = torch.cuda.Stream(device=dev)
        torch.cuda.set_stream(stream)
        res = {}

        def shard_wants(model, x, n_local):
            """this process's own reconstruct_dev of every rank's shard, at the shard size"""
            out = []
            for r in range(world):
                w = torch.empty(n_local, 3, 64, 64, device=dev)
                model.reconstruct_dev(x[r * n_local:(r + 1) * n_local].data_ptr(), n_local, 0, w.data_ptr(), stream.cuda_stream)
                out.append(w)
            return out

        def mismatch(got, wants, n_local):
            """device bool, enqueued on the stream: does any rank's slot differ from its local result in any bit"""
            return torch.stack([(got[r * n_local:(r + 1) * n_local] != wants[r]).any() for r in range(world)]).any()

        for graph in GRAPHS:
            W = _weights(graph)
            for n_local in (5, 64):                       # 5: small-batch split-K schedule; 64: the CTA-pair kernel
                model = pkg.IAN(graph, True, weights=W, device=rank)
                model.setup_fused_gather(n_local)
                n = n_local * world
                lo = rank * n_local
                for precision in ("fp32", "bf16"):
                    model.set_precision(precision)
                    for form, pipelined in (("fused", False), ("pipelined", True)):
                        ok = True
                        for t in range(4):
                            x = _images(100 * t + 7, n, dev)
                            wants = shard_wants(model, x, n_local)
                            if (t + rank) % 2 == 0:
                                torch.cuda._sleep(int(4e8))       # ~0.2 s of device-side delay on alternating ranks
                            shard = x[lo:lo + n_local].contiguous()
                            if pipelined:
                                model.reconstruct_gather_async_dev(shard.data_ptr(), n_local, 0, stream.cuda_stream)
                                ptr = model.gather_wait_dev(stream.cuda_stream)
                            else:
                                ptr = model.reconstruct_gather_dev(shard.data_ptr(), n_local, 0, stream.cuda_stream)
                            got = par.as_cuda_tensor(ptr, (n, 3, 64, 64), dev)
                            bad = mismatch(got, wants, n_local)   # consumer enqueued in stream order BEFORE the next call
                            if (t + rank) % 2 == 1:
                                torch.cuda._sleep(int(2e8))       # ... and the slow consumer side of the skew
                            ok = ok and not bool(bad.item())
                        res["%s_n%d_%s_%s" % (graph, n_local, precision, form)] = ok
                model.close()

        # the public sharded entry, a shard of one 512-image chunk plus one 8-image chunk
        n_local = 520
        n = n_local * world
        model = pkg.IAN("IAN.py", True, weights=_weights("IAN.py"), device=rank)
        model.set_precision("bf16")
        x = _images(5, n, dev)
        wants = shard_wants(model, x, n_local)
        for form, pipelined in (("fused", False), ("pipelined", True)):
            got = model.reconstruct_sharded(x, stream=stream.cuda_stream, pipelined=pipelined)
            res["IAN.py_sharded_520_bf16_%s" % form] = not bool(mismatch(got, wants, n_local).item())
        torch.cuda.synchronize()
        model.close()
        dist.destroy_process_group()
        q.put((rank, res, None))
    except Exception:
        q.put((rank, None, traceback.format_exc()))


def test_two_gpu_flow_gather_bit_identical_with_rank_skew():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    out = [q.get(timeout=900) for _ in procs]
    for p in procs:
        p.join(timeout=120)
    if os.environ.get("IAN_TEST_RECORD"):
        import json
        os.makedirs(os.environ["IAN_TEST_RECORD"], exist_ok=True)
        with open(os.path.join(os.environ["IAN_TEST_RECORD"], "two_gpu_gather_flow.json"), "w") as f:
            json.dump({str(r): (res if err is None else err) for r, res, err in out}, f, indent=1)
    for rank, res, err in out:
        assert err is None, "rank %d:\n%s" % (rank, err)
        bad = [tag for tag, ok in res.items() if not ok]
        assert not bad, (rank, bad)
