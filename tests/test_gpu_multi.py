"""Read-sharded locus on TWO GPUs (SURVEY.md 8e): every rank types its half of the reads of one unit - pileup counts
all-reduced before the representative-base sets are derived, class tables merged so that every class lives on one rank,
EM as one cooperative kernel per rank that sums through NVLink peer memory (em_dist.py) - and the union must equal the
unsharded run on one GPU: read / pair totals, the merged class table (by allele set), identical ranked alleles on both ranks,
abundances within 1e-6.  Needs >= 2 visible GPUs (skipped otherwise)."""
import os
import pickle
import socket
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _case():
    from helpers import synthetic_case
    args, sam, truth = synthetic_case(29, A=700, L=2500, n_pairs=3000, base="ov", del_frac=0.1, paired=False)
    return args, sam


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import torch
    import torch.distributed as dist
    import _hgt_path
    _hgt_path.load()
    from hisatgenotype_b200 import typing_core as TC
    from hisatgenotype_b200.locus import LocusTables
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    args, sam = _case()
    t = LocusTables(*args, device=rank)
    mine = sam[rank * len(sam) // world:(rank + 1) * len(sam) // world]  # contiguous shard of the name-sorted text
    bt = TC.Batch([t], TC.make_params(allow_discordant=True), True, device=rank)
    bt.set_pileup_allreduce()
    bt.set_skip_em(True)
    bt.add_unit(0, mine)
    bt.run()
    # default: tables merged (every class on one rank) + ONE cooperative kernel per rank summing through NVLink peer memory
    ranked, iters = bt.sharded_abundance(0)
    ranked_again, iters_again = bt.sharded_abundance(0)  # second launch on the same exchange blocks
    peer_classes = bt.shard_ms["classes"]
    assert bt.shard_ms["em"] == "peer"
    s = bt.unit_summary(0)
    res = {"reads": s["num_reads"], "pairs": s["num_pairs"], "cmpt": bt.unit_gene_cmpt(0, TC.TABLE_GENE), "ranked": ranked,
           "iters": iters, "ranked_again": ranked_again, "iters_again": iters_again, "peer_classes": peer_classes}
    with open(os.path.join(out_dir, "rank%d.pkl" % rank), "wb") as f:
        pickle.dump(res, f)
    bt.close()
    t.close()
    dist.barrier()
    dist.destroy_process_group()


def test_two_gpu_read_sharded_locus_equals_unsharded(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    shards = [pickle.load(open(os.path.join(str(tmp_path), "rank%d.pkl" % r), "rb")) for r in range(2)]
    # the unsharded run
    from hisatgenotype_b200 import typing_core as TC
    from hisatgenotype_b200.locus import LocusTables
    args, sam = _case()
    t = LocusTables(*args)
    bt = TC.Batch([t], TC.make_params(allow_discordant=True), True)
    bt.add_unit(0, sam)
    bt.run()
    s = bt.unit_summary(0)
    assert shards[0]["reads"] + shards[1]["reads"] == s["num_reads"]
    assert shards[0]["pairs"] + shards[1]["pairs"] == s["num_pairs"]
    merged = {}
    for sh in shards:
        for k, c in sh["cmpt"].items():
            merged[k] = merged.get(k, 0) + c
    assert merged == bt.unit_gene_cmpt(0, TC.TABLE_GENE)
    whole = bt.unit_abundance(0)
    assert shards[0]["ranked"] == shards[1]["ranked"] and shards[0]["iters"] == shards[1]["iters"]
    assert [a for a, _ in shards[0]["ranked"]] == [a for a, _ in whole]
    for (_, x), (_, y) in zip(shards[0]["ranked"], whole):
        assert x == pytest.approx(y, rel=1e-6, abs=1e-12)
    assert shards[0]["iters"] == s["em_iters"][0]
    for sh in shards:
        assert sh["ranked_again"] == sh["ranked"] and sh["iters_again"] == sh["iters"]
    # after the merge every class lives on exactly one rank
    assert shards[0]["peer_classes"] + shards[1]["peer_classes"] == len(merged)
    bt.close()
    t.close()
