"""The sharded path behind the C ABI (hx_shard_group_*): local search into the send block, ONE ncclAllGather issued by the
library, (score, id) merge.  A group of one runs everywhere; the two-rank test needs two devices and skips on one."""
import os
import socket
import sys
from pathlib import Path

import numpy as np
import pytest

import helix_db_b200 as hx
from helix_db_b200 import sharding as sh
from oracle import hxo
from test_gpu_parity import build_pair

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent


def test_group_of_one_matches_unsharded():
    rng = np.random.default_rng(5)
    n, dim, B, k = 3000, 48, 200, 10
    rows = rng.standard_normal((n, dim)).astype(np.float32)
    gpu, ora = build_pair(hx.Metric.Cosine, hxo.COSINE, rows, m=8, m0=16, efc=60)
    q = rng.standard_normal((B, dim)).astype(np.float32)
    g = sh.ShardGroup(gpu, 1, 0, None)
    p = hx.SearchParams.strict(k, 50)
    ids, sc, cnt = g.search(sh.HNSW, q, p, k)
    oi, os_, oc, _, _ = ora.search_batch(q, k, 50, threads=4)
    assert cnt.tolist() == oc.tolist() and ids.tolist() == oi.tolist() and sc.tobytes() == os_.tobytes()
    # per-shard k above k_out: the merge truncates
    ids2, sc2, cnt2 = g.search(sh.HNSW, q, hx.SearchParams.strict(20, 50), k)
    assert ids2.tolist() == oi.tolist() and sc2.tobytes() == os_.tobytes()
    cand = np.arange(0, n, 3, dtype=np.uint64)
    rids, rsc, rcnt = g.search_restricted(q[:30], hx.SearchParams.strict(k), cand)
    for b in range(30):
        ei, es = ora.search_restricted(q[b], k, cand)
        assert rids[b, :rcnt[b]].tolist() == ei.tolist() and rsc[b, :rcnt[b]].tobytes() == es.tobytes()
    local_ms, coll_ms = g.last_ms()
    assert local_ms > 0.0
    g.close()
    gpu.close()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _rank_main(rank, world, port, ret):
    sys.path.insert(0, str(ROOT))
    sys.path.insert(0, str(ROOT / "tests"))
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)      # host channel for the unique id only
    torch.cuda.set_device(rank)
    import helix_db_b200 as hx2
    from helix_db_b200 import sharding as sh2
    from oracle import hxo as o2
    from hx_testutil import mirror_from_oracle
    from test_gpu_parity import levels_for

    rng = np.random.default_rng(77)                                   # same data on every rank
    n, dim, B, k = 4000, 64, 300, 10
    rows = rng.standard_normal((n, dim)).astype(np.float32)
    q = rng.standard_normal((B, dim)).astype(np.float32)
    ids = np.arange(500, 500 + n, dtype=np.uint64)
    # every rank builds EVERY shard's oracle (to state the expected merged answer); it mirrors only its own onto its GPU
    oras = []
    for r in range(world):
        lo, hi = sh2.shard_range(n, world, r)
        o = o2.Index(o2.EUCLIDEAN, dim, m=8, m0=16, ef_construction=60)
        for i, lv in zip(range(lo, hi), levels_for(hi - lo, 8, 100 + r)):
            o.insert(int(ids[i]), rows[i], lv)
        oras.append(o)
    gpu = hx2.VectorIndex(hx2.Metric.Euclidean, hx2.VectorIndexConfig("s", "embedding", dim).with_m(8).with_m0(16)
                          .with_ef_construction(60), device=rank, storage=1)
    mirror_from_oracle(gpu, oras[rank])
    uid = sh2.exchange_unique_id(rank)
    g = sh2.ShardGroup(gpu, world, rank, uid)
    # HNSW path: expected = (score, id) merge of the oracles' per-shard answers over the identical per-shard graphs
    ef = 40
    got_i, got_s, got_c = g.search(sh2.HNSW, q, hx2.SearchParams.strict(k, ef), k)
    for b in range(B):
        items = []
        for o in oras:
            oi, os_ = o.search(q[b], k, ef=ef)
            items += [(np.float32(s).view(np.uint32).item(), int(i)) for i, s in zip(oi, os_)]
        items.sort()
        items = items[:k]
        assert got_c[b] == len(items) and got_i[b, :got_c[b]].tolist() == [i for _, i in items], f"rank {rank} query {b}"
        assert got_s[b, :got_c[b]].view(np.uint32).tolist() == [s for s, _ in items]
    # exhaustive tensor-core path and restricted path: exact => equal to the unsharded oracle, whatever the sharding
    full = o2.Index(o2.EUCLIDEAN, dim)
    full.put_vectors(ids, rows)
    full.set_entry(int(ids[0]), 0)
    d_i, d_s, d_c = g.search(sh2.DENSE, q[:64], hx2.SearchParams.strict(k), k)
    cand = ids[::5].copy()
    r_i, r_s, r_c = g.search_restricted(q[:64], hx2.SearchParams.strict(k), cand)
    for b in range(64):
        ei, es = full.search_exact(q[b], k)
        assert d_i[b, :d_c[b]].tolist() == ei.tolist() and d_s[b, :d_c[b]].tobytes() == es.tobytes()
        ri, rs = full.search_restricted(q[b], k, cand)
        assert r_i[b, :r_c[b]].tolist() == ri.tolist() and r_s[b, :r_c[b]].tobytes() == rs.tobytes()
    dist.barrier()
    g.close()
    gpu.close()
    dist.destroy_process_group()
    ret[rank] = True


def test_two_ranks_one_all_gather():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    import torch.multiprocessing as mp
    world, port = 2, _free_port()
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_rank_main, args=(world, port, ret), nprocs=world, join=True)
    assert all(ret.get(r) for r in range(world))
