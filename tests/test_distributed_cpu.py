"""N > 1 host logic on CPU (gloo, world_size 2).

The CUDA path cannot run here, so this checks what surrounds it: the slab partition, the
id exchange over torch.distributed, and -- with the REFERENCE's own C accelerator driven
through its `dp` hook by a gloo all-reduce (oracle/_ref, when built; else the port, pinned
bit-identical to it, through the same hook) -- that "each rank updates its slab, dot products
are summed over ranks" reproduces the serial full-vector update exactly as the reference
promises (src-F08-vector/README.md:16-22).  That is the contract libnka_b200's NCCL path
implements on the GPUs (checked for real by tests/test_gpu_multi.py)."""
import os
import socket
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_slab_bounds_partition():
    from nka_b200.distributed import slab_bounds
    for n in (0, 1, 2, 3, 7, 16, 1001, 1 << 20, (1 << 28) + 5):
        for world in (1, 2, 3, 4, 8):
            edges = [slab_bounds(n, world, r) for r in range(world)]
            assert edges[0][0] == 0 and edges[-1][1] == n
            for (a, b), (c, d) in zip(edges, edges[1:]):
                assert b == c and a <= b
            assert all(lo % 2 == 0 for lo, _ in edges)
            sizes = [b - a for a, b in edges]
            assert max(sizes) - min(sizes) <= 2 or n < 2 * world
    with pytest.raises(ValueError):
        slab_bounds(10, 2, 2)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _worker(rank, world, port, n, mvec, q):
    import ctypes as C
    import torch
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from nka_b200.distributed import exchange_unique_id, slab_bounds
    from oracle import api
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        uid = exchange_unique_id()
        lo, hi = slab_bounds(n, world, rank)
        lib = api.ref_lib()
        flags = [None] * world
        dist.all_gather_object(flags, lib is not None)
        results = {"uid": uid, "bounds": (lo, hi), "impl": "reference" if all(flags) else "port"}

        def global_dot(length, x, y):
            a = np.ctypeslib.as_array(x, shape=(length,)) if length else np.zeros(0)
            b = np.ctypeslib.as_array(y, shape=(length,)) if length else np.zeros(0)
            t = torch.tensor([float(np.dot(a, b))], dtype=torch.float64)
            dist.all_reduce(t)
            return float(t.item())

        cb = api.DP_FUNC(global_dot)
        if all(flags):
            h = lib.nka_init(hi - lo, mvec, 0.01, C.cast(cb, C.c_void_p))
            update = lambda f: lib.nka_accel_update(h, f.ctypes.data_as(C.POINTER(C.c_double)))
            num_vec = lambda: lib.nka_num_vec(h)
        else:
            # without the compiled reference: the port, which routes every dot product through the same hook
            acc = api.OracleNKA(hi - lo, mvec, 0.01, dp=cb)
            update, num_vec = acc.accel_update, acc.num_vec
        rng = np.random.default_rng(77)
        outs, nvec = [], []
        for t in range(mvec + 5):
            full = rng.uniform(-0.5, 0.5, n) * 0.8 ** t
            mine = np.ascontiguousarray(full[lo:hi])
            update(mine)
            outs.append(mine)
            nvec.append(num_vec())
        if all(flags):
            lib.nka_delete(h)
        else:
            acc.close()
        results["outs"] = outs
        results["nvec"] = nvec
        q.put((rank, results))
    finally:
        dist.destroy_process_group()


def test_two_rank_slab_update_equals_serial_update():
    import torch.multiprocessing as mp
    from oracle import api
    n, mvec, world = 1001, 4, 2
    api.oracle_lib()            # built here, once: two ranks compiling it at the same time could load a partial file
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, n, mvec, q)) for r in range(world)]
    for p in procs:
        p.start()
    got = dict(q.get(timeout=120) for _ in range(world))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    # the 128-byte id reached both ranks unchanged
    assert got[0]["uid"] == got[1]["uid"] and len(got[0]["uid"]) == 128
    assert got[0]["bounds"][1] == got[1]["bounds"][0]
    assert got[0]["impl"] == got[1]["impl"]
    # serial reference on the full vectors (long-double dots: summation order differs across the split)
    ser = api.OracleNKA(n, mvec, 0.01, dotmode=1)
    rng = np.random.default_rng(77)
    for t in range(mvec + 5):
        full = rng.uniform(-0.5, 0.5, n) * 0.8 ** t
        ser.accel_update(full)
        joined = np.concatenate([got[0]["outs"][t], got[1]["outs"][t]])
        assert np.linalg.norm(joined - full) <= 1e-12 * np.linalg.norm(full), t
        assert got[0]["nvec"][t] == got[1]["nvec"][t] == ser.num_vec()


def test_row_slabs_tile_the_grid():
    """nka_b200.example.row_slab: contiguous, balanced, complete (the slab example's partition)."""
    from nka_b200.example import row_slab
    for ny in (9, 50, 64, 131, 4096, 32768):
        for world in (1, 2, 3, 4, 8):
            if ny // world < 3:
                continue
            bounds = [row_slab(ny, world, r) for r in range(world)]
            assert bounds[0][0] == 0 and bounds[-1][1] == ny
            assert all(bounds[r][1] == bounds[r + 1][0] for r in range(world - 1))
            sizes = [b - a for a, b in bounds]
            assert min(sizes) >= 3 and max(sizes) - min(sizes) <= 1
