"""world_size-2 (and 3) gloo test of the N>1 path's host logic: equal-pair row shards + one all-gather of the
row blocks reproduce the full packed triangle.  The per-rank compute is the oracle here (no GPU in this tier)."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from famsa_b200 import seqio, sharding
from oracle import pyoracle


def _worker(rank, world, port, n, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    codes, offsets, lens = seqio.synth_family(n, 60, seed=4)
    bounds = sharding.row_shards(n, world)
    rb, re = bounds[rank], bounds[rank + 1]
    sizes = sharding.shard_sizes(bounds)
    block = torch.zeros(max(sizes), dtype=torch.int16)
    mine = pyoracle.lcs_triangle(codes, offsets, lens, rb, re).astype(np.int16)
    block[:mine.size] = torch.from_numpy(mine)
    gathered = sharding.all_gather_blocks(block, bounds, dist)
    full = sharding.full_triangle(gathered, bounds).numpy().astype(np.uint32)
    want = pyoracle.lcs_triangle(codes, offsets, lens)
    ok = np.array_equal(full, want) and sum(sizes) == want.size
    open(os.path.join(out_dir, f"rank{rank}.txt"), "w").write("ok" if ok else "bad")
    dist.destroy_process_group()


def _pipelined_worker(rank, world, port, n, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    codes, offsets, lens = seqio.synth_family(n, 60, seed=4)
    bounds = sharding.row_shards(n, world)
    full = torch.full((sharding.tri(n),), -1, dtype=torch.int16)

    def compute_rows(r0, r1, view):
        view.copy_(torch.from_numpy(pyoracle.lcs_triangle(codes, offsets, lens, r0, r1).astype(np.int16)))
    sharding.triangle_allgather_pipelined(compute_rows, bounds, rank, dist, full, n_sub=3)
    want = pyoracle.lcs_triangle(codes, offsets, lens)
    ok = np.array_equal(full.numpy().astype(np.uint32), want)
    open(os.path.join(out_dir, f"rank{rank}.txt"), "w").write("ok" if ok else "bad")
    dist.destroy_process_group()


@pytest.mark.parametrize("world,n", [(2, 101), (3, 64), (2, 3)])
def test_pipelined_all_gather(tmp_path, world, n):
    """Row shards cut into pieces, every piece broadcast into its place of the full packed triangle (the overlapped
    exchange of the N>1 bench path) -- host logic on gloo, compute by the oracle."""
    port = 29700 + world * 7 + (os.getpid() % 50)
    mp.spawn(_pipelined_worker, args=(world, port, n, str(tmp_path)), nprocs=world, join=True)
    for r in range(world):
        assert open(tmp_path / f"rank{r}.txt").read() == "ok"


def _assign_worker(rank, world, port, n, out_dir):
    """Host logic of the sharded medoid assignment on gloo: per-shard packed results (computed by the oracle here),
    one MIN all-reduce, unpack == the sequential loop over all seeds."""
    from famsa_b200.binding import unpack_assignment
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    codes, offsets, lens = seqio.synth_family(n, 50, seed=9, sort_desc=False)
    seeds = np.array([3, 17, 5, 3, n - 1], dtype=np.uint32)          # a repeated seed: ties must go to the first
    rows = pyoracle.lcs_rows(codes, offsets, lens, seeds)
    dmat = np.array([[pyoracle.transform(0, int(rows[k, j]), int(lens[seeds[k]]), int(lens[j]), False) for j in range(n)]
                     for k in range(len(seeds))], dtype=np.float32)
    want_a = np.zeros(n, dtype=np.uint32); want_d = dmat[0].copy()
    for k in range(1, len(seeds)):                                   # FastTree.cpp:317-322, strict <
        better = dmat[k] < want_d
        want_a[better] = k; want_d[better] = dmat[k][better]
    order = np.argsort(-lens.astype(np.int64), kind="stable")        # famsa_lcs_upload's length-descending order
    pos = np.empty(n, dtype=np.int64); pos[order] = np.arange(n)

    def assign_shard(shard, n_shards, packed):
        g0, g1 = sharding.group_slice((n + 31) // 32, shard, n_shards)
        mine = (pos // 32 >= g0) & (pos // 32 < g1)
        p = np.full(n, np.iinfo(np.int64).max, dtype=np.int64)
        p[mine] = (want_d[mine].view(np.uint32).astype(np.int64) << 32) | want_a[mine].astype(np.int64)
        packed.copy_(torch.from_numpy(p))
    packed = torch.empty(n, dtype=torch.int64)
    sharding.assign_allreduce(assign_shard, packed, rank, world, dist)
    a, d = unpack_assignment(packed.numpy())
    ok = np.array_equal(a, want_a) and np.array_equal(d, want_d)
    open(os.path.join(out_dir, f"rank{rank}.txt"), "w").write("ok" if ok else "bad")
    dist.destroy_process_group()


@pytest.mark.parametrize("world,n", [(2, 150), (3, 70)])
def test_sharded_assignment_allreduce(tmp_path, world, n):
    port = 29800 + world * 7 + (os.getpid() % 50)
    mp.spawn(_assign_worker, args=(world, port, n, str(tmp_path)), nprocs=world, join=True)
    for r in range(world):
        assert open(tmp_path / f"rank{r}.txt").read() == "ok"


def test_sub_bounds():
    for rb, re, k in [(0, 1000, 4), (700, 1000, 4), (5, 6, 4), (0, 0, 3), (0, 2, 8)]:
        b = sharding.sub_bounds(rb, re, k)
        assert b[0] == rb and b[-1] == re and len(b) == k + 1 and all(x <= y for x, y in zip(b, b[1:]))


@pytest.mark.parametrize("world,n", [(2, 101), (3, 64)])
def test_row_shards_all_gather(tmp_path, world, n):
    port = 29600 + world * 7 + (os.getpid() % 50)
    mp.spawn(_worker, args=(world, port, n, str(tmp_path)), nprocs=world, join=True)
    for r in range(world):
        assert open(tmp_path / f"rank{r}.txt").read() == "ok"


def test_row_shards_balance():
    for n, parts in [(10000, 2), (20000, 4), (28284, 8), (7, 8), (1, 2)]:
        b = sharding.row_shards(n, parts)
        assert b[0] == 0 and b[-1] == n and all(x <= y for x, y in zip(b, b[1:]))
        sizes = sharding.shard_sizes(b)
        assert sum(sizes) == n * (n - 1) // 2
        if n >= 1000:
            # boundaries sit on 32-row mask groups (the kernel's unit of work: a group split between two ranks is computed by both)
            assert max(sizes) <= 1.02 * (sum(sizes) / parts)
            assert all(x % 32 == 0 for x in b[1:-1])


def test_schedule_levels_and_shards():
    from famsa_b200.schedule import ready_levels, shard_level
    merges = [(0, 1), (2, 3), (4, 5), (6, 7), (8, 9)]        # 6 leaves: (0,1)->6 (2,3)->7 (4,5)->8 (6,7)->9 (8,9)->10
    lv = ready_levels(6, merges)
    assert lv == [[0, 1, 2], [3], [4]]
    parts = shard_level([0, 1, 2, 3], [10, 7, 5, 4], 2)
    assert sorted(sum(parts, [])) == [0, 1, 2, 3] and abs(sum([10, 7, 5, 4][k] for k in parts[0]) - 13) <= 3


def _tree_worker(rank, world, port, n, out_dir):
    import sys
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from dp_cases import OracleEngine, random_tree
    from famsa_b200 import schedule
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    z = np.load(os.path.join(out_dir, "case.npz"))
    seqs = [str(s) for s in z["seqs"]]
    merges = [tuple(int(x) for x in m) for m in z["merges"]]
    codes, off, lens = seqio.pack([seqio.encode(s) for s in seqs])
    eng = OracleEngine()
    eng.upload(codes, off, lens)
    eng.prof_set_scoring(z["sm"])
    results, root = schedule.sharded_resident_alignment(eng, dist, rank, world, len(seqs), lens, merges, z["gaps"])
    everything = [None] * world
    dist.all_gather_object(everything, {k: (r["path"], r["swapped"], r["total"]) for k, r in results.items()})
    if rank == 0:
        merged = {}
        for part in everything:
            assert not (set(part) & set(merged)), "a merge ran on two ranks"
            merged.update(part)
        np.savez(os.path.join(out_dir, "out.npz"), keys=np.array(sorted(merged)),
                 **{f"p{k}": merged[k][0] for k in merged}, sw=np.array([merged[k][1] for k in sorted(merged)]),
                 tot=np.array([merged[k][2] for k in sorted(merged)]), n_ranks_with_work=sum(1 for p in everything if p),
                 live=len(eng.tab), root=root)
    else:
        assert root is None and not eng.tab, "non-root ranks must hand everything over"
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_subtree_sharded_resident_alignment(tmp_path, world):
    """HP-2 on several ranks with resident profiles: whole subtrees per rank (no communication), subtree roots handed
    to rank 0, top merges there.  Every merge runs exactly once and the assembled alignment is the reference's."""
    import sys
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from dp_cases import assemble_rows, random_tree, reference_merges, reference_score_matrix
    n = 26
    rng = np.random.default_rng(8)
    codes, off, lens = seqio.synth_family(n, 45, 8, sort_desc=False)
    seqs = [seqio.decode(codes[int(o):int(o) + int(l)]) for o, l in zip(off, lens)]
    merges = random_tree(n, rng, 0.3)
    g, recs = reference_merges(seqs, merges, threads=(1,))
    sm = reference_score_matrix(n)
    np.savez(tmp_path / "case.npz", seqs=np.array(seqs), merges=np.array(merges), sm=sm, gaps=g)
    port = 29640 + world
    mp.spawn(_tree_worker, args=(world, port, n, str(tmp_path)), nprocs=world, join=True)
    z = np.load(tmp_path / "out.npz")
    assert list(z["keys"]) == list(range(len(merges))) and int(z["n_ranks_with_work"]) == world
    assert int(z["live"]) == 1
    results = {int(k): dict(path=z[f"p{k}"], swapped=bool(s), total=int(t)) for k, s, t in zip(z["keys"], z["sw"], z["tot"])}
    assert [results[k]["total"] for k in range(len(merges))] == [r["total"] for r in recs]
    assert assemble_rows(seqs, merges, results) == recs[-1]["rows"]


@pytest.mark.parametrize("n,world,cat", [(2, 2, 0.0), (3, 4, 0.0), (40, 2, 0.9), (333, 4, 0.3), (1000, 8, 0.05), (64, 3, 1.0)])
def test_subtree_shards_properties(n, world, cat):
    """Every merge has exactly one executor; a subtree below a frontier node stays on that node's rank (so both children
    of every sharded merge are local); top merges only combine frontier nodes or other top merges; loads are balanced."""
    import sys
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from dp_cases import random_tree
    from famsa_b200.schedule import ready_levels_subset, subtree_shards
    merges = random_tree(n, np.random.default_rng(n + world), cat)
    owner, frontier = subtree_shards(n, merges, world)
    assert len(owner) == len(merges) and all(-1 <= o < world for o in owner)
    fr = dict(frontier)
    node_rank = {}
    for k, (a, b) in enumerate(merges):
        v = n + k
        if owner[k] >= 0:
            for c in (a, b):                     # children are leaves or merges of the same rank
                assert c < n or owner[c - n] == owner[k]
            node_rank[v] = owner[k]
        else:
            assert v not in fr
            for c in (a, b):                     # a top merge consumes frontier nodes or other top merges
                assert c in fr or (c >= n and owner[c - n] == -1)
    assert all((v < n) or owner[v - n] == r for v, r in frontier)
    # the frontier partitions the leaves
    leaves_under = {}
    for i in range(n):
        leaves_under[i] = {i}
    for k, (a, b) in enumerate(merges):
        leaves_under[n + k] = leaves_under[a] | leaves_under[b]
    covered = [leaf for v, _ in frontier for leaf in leaves_under[v]]
    assert sorted(covered) == list(range(n))
    loads = [sum(1 for o in owner if o == r) for r in range(world)]
    if n >= 50 * world:
        assert max(loads) <= 1.25 * sum(loads) / world + 4       # LPT over ~4 pieces per rank
    # levels of a rank's subset respect dependencies
    for r in range(world):
        done = set()
        for lvl in ready_levels_subset(n, merges, [k for k in range(len(merges)) if owner[k] == r]):
            for k in lvl:
                for c in merges[k]:
                    assert c < n or (c - n) in done
            done.update(lvl)
