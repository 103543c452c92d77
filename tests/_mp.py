"""Helpers to run a function on several ranks (one process per rank, env:// rendezvous on 127.0.0.1)."""
import os
import socket
import sys
import traceback

import torch
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _worker(rank, world, port, backend, fn, args, ret, extra_env):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank), LOCAL_WORLD_SIZE=str(world), DEAR_BACKEND=backend)
    os.environ.update(extra_env or {})
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    torch.set_num_threads(1)
    try:
        import dear_pytorch_b200 as dear
        dear.init()
        out = fn(rank, world, *args)
        dear.shutdown()
        ret[rank] = ("ok", out)
    except Exception:
        ret[rank] = ("err", traceback.format_exc())
        raise


def run_ranks(fn, world=2, backend="gloo", args=(), timeout=240, extra_env=None, start_method=None):
    """Run ``fn(rank, world, *args)`` on ``world`` processes; returns the list of results.

    CPU backends start their ranks from a fork server that has imported torch but never run autograd (~10x faster
    than spawn).  Forking the test process itself is not safe: once it has run a backward pass on a machine with a
    GPU, autograd's per-device worker threads exist and a forked child's backward raises.  Anything touching CUDA
    must spawn.  Either way ``fn`` and ``args`` are pickled, so ``fn`` must be a module-level function.
    """
    if start_method is None:
        start_method = "forkserver" if backend in ("gloo", "emu") else "spawn"
    ctx = mp.get_context(start_method)
    if start_method == "forkserver":
        # takes effect when the (per test session) server starts; the first torch.optim optimizer of a process imports
        # torch._dynamo, which costs seconds per rank unless the server did it once
        ctx.set_forkserver_preload(["torch", "torch._dynamo"])
    mgr = ctx.Manager()
    ret = mgr.dict()
    port = free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, backend, fn, args, ret, extra_env)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout)
    alive = [p for p in procs if p.is_alive()]
    for p in alive:
        p.terminate()
    if alive:
        raise RuntimeError("ranks hung (timeout %ss): %s" % (timeout, dict(ret)))
    res = dict(ret)
    errs = {r: v[1] for r, v in res.items() if v[0] == "err"}
    if errs or len(res) != world:
        raise RuntimeError("rank failures: %s" % (errs or res))
    return [res[r][1] for r in range(world)]
