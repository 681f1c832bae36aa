"""Spawn `world` processes running `fn(rank, world, *args)` with a gloo
rendezvous on 127.0.0.1 and return the per-rank results."""
import os
import pickle
import socket
import tempfile
import traceback

import torch.multiprocessing as mp


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _entry(rank, world, port, fn, args, outdir, env):
    # the ranks are CPU processes: with a GPU visible every rank would pick NCCL on the
    # same device, which NCCL refuses (CUDA is first initialised after this line)
    os.environ.update({"RANK": str(rank), "WORLD_SIZE": str(world),
                       "LOCAL_RANK": str(rank), "MASTER_ADDR": "127.0.0.1",
                       "MASTER_PORT": str(port), "OMP_NUM_THREADS": "1",
                       "CUDA_VISIBLE_DEVICES": ""})
    os.environ.update(env or {})
    import torch
    torch.set_num_threads(1)
    try:
        res = ("ok", fn(rank, world, *args))
    except Exception:
        res = ("err", traceback.format_exc())
    with open(os.path.join(outdir, "r%d.pkl" % rank), "wb") as f:
        pickle.dump(res, f)
    try:
        import torch.distributed as dist
        if dist.is_initialized():
            dist.destroy_process_group()
    except Exception:
        pass


def run_distributed(fn, world, *args, env=None, timeout=240):
    port = _free_port()
    with tempfile.TemporaryDirectory() as d:
        ctx = mp.get_context("spawn")
        procs = [ctx.Process(target=_entry,
                             args=(r, world, port, fn, args, d, env))
                 for r in range(world)]
        for p in procs:
            p.start()
        for p in procs:
            p.join(timeout)
        for p in procs:
            if p.is_alive():
                p.kill()
                raise RuntimeError("distributed test timed out")
        out = []
        for r in range(world):
            fn_ = os.path.join(d, "r%d.pkl" % r)
            if not os.path.exists(fn_):
                raise RuntimeError("rank %d produced no result (exit %s)"
                                   % (r, procs[r].exitcode))
            with open(fn_, "rb") as f:
                status, val = pickle.load(f)
            if status != "ok":
                raise RuntimeError("rank %d failed:\n%s" % (r, val))
            out.append(val)
        return out
