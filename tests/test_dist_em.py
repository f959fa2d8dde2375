"""The class-table exchange of the read-sharded EM (hisat-genotype_b200/em_dist.py) under gloo, world_size 2, CPU only.

gather_class_tables is the all_gather in front of hgt_class_merge_dev; the merge and the peer-memory EM behind it need
GPUs (tests/test_gpu_em.py, tests/test_gpu_multi.py)."""
import os
import socket
import sys

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _gather_worker(rank, world, port, out):
    sys.path.insert(0, ROOT)
    import _hgt_path
    _hgt_path.load()
    from hisatgenotype_b200 import em_dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    wp = 4
    res = []
    for sizes in ((3, 5), (0, 4), (6, 0), (0, 0)):  # ragged and empty shards
        n = sizes[rank]
        rng = np.random.default_rng(100 * rank + n)
        bits = torch.from_numpy(rng.integers(0, 1 << 62, size=n * wp, dtype=np.int64))
        cnt = torch.from_numpy(rng.integers(1, 50, size=n, dtype=np.int64))
        first = torch.from_numpy((np.arange(n, dtype=np.int32) * 3 + 1000 * rank).astype(np.int32))
        g = em_dist.gather_class_tables(bits, cnt, first, wp)
        res.append((bits.numpy().copy(), cnt.numpy().copy(), first.numpy().copy(), [x.numpy().copy() if hasattr(x, "numpy") else x for x in g]))
    out.put((rank, res))
    dist.barrier()
    dist.destroy_process_group()


def test_gather_class_tables_ragged_world2():
    """The table exchange in front of hgt_class_merge_dev (em_dist.gather_class_tables) under gloo: every rank obtains the
    concatenation of all ranks' rows / counts / first indices in rank order, whatever the shard sizes (also empty ones)."""
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    procs = [ctx.Process(target=_gather_worker, args=(r, 2, port, out)) for r in range(2)]
    for p in procs:
        p.start()
    got = dict(out.get(timeout=120) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for case in range(4):
        want_bits = np.concatenate([got[r][case][0] for r in range(2)])
        want_cnt = np.concatenate([got[r][case][1] for r in range(2)])
        want_first = np.concatenate([got[r][case][2] for r in range(2)])
        for r in range(2):
            g_bits, g_cnt, g_first, n_total = got[r][case][3]
            assert n_total == len(want_cnt)
            np.testing.assert_array_equal(g_bits, want_bits)
            np.testing.assert_array_equal(g_cnt, want_cnt)
            np.testing.assert_array_equal(g_first, want_first)
