#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on BASELINE.json's configuration.

A "step" is one pass of the hot path over one batch: the all-pairs LCS triangle of a synthetic
protein family (SURVEY.md section 8(d) generator).
  N = 1 : configs[1] -- 10 000 proteins x 400 aa, 49 995 000 LCS lengths on one B200.
  N > 1 : the same per-GPU work ("weak"): 10 000*sqrt(N) proteins, triangle rows sharded so that every
          rank owns the same number of pairs, then ONE NCCL all-gather of the uint16 row blocks
          (the north star's "final all-gather of the distance row blocks").
value   = LCS pairs / s, inputs (residue codes + bit-mask tables) resident in HBM, results left in HBM.
e2e     = the same metric through the host-buffer C ABI call a FAMSA guide-tree builder would make
          (famsa_lcs_upload + famsa_lcs_triangle): H2D of the residues, mask build, kernel, D2H of
          the triangle -- all inside the timed region, every step.
--impl reference : the UNMODIFIED reference (oracle/_ref: CLCSBP AVX2 path driven by the reference's
          own calculateDistanceVector, UPGMA's row-parallel shape) on all host threads, same config.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_BASE, LEN, SEED = 10000, 400, 1
METRIC = "pairwise LCS distances/sec"
UNIT = "pairs/s"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def workload(n_gpus: int):
    from famsa_b200 import seqio
    n = int(round(N_BASE * math.sqrt(n_gpus)))
    return seqio.synth_family(n, LEN, SEED), n


from famsa_b200.sharding import (row_shards, shard_sizes, tri, PeerTriangle, assign_allreduce)  # noqa: E402


def config_for(n: int, world: int) -> dict:
    """The `config` object of the JSON line -- identical in the b200 arm and in --impl reference."""
    return {"workload": f"LCS triangle, {n} x {LEN} aa synthetic family (seed {SEED})",
            "n_seqs": n, "len": LEN, "pairs_per_step": tri(n),
            "out": "uint16 packed lower triangle", "l2": "flushed between timed iterations (192 MiB write)",
            "multi_gpu": ("row shards with equal pairs, each computed in 8 pieces; every finished piece is copied into its place of "
                          "every peer's full packed triangle (CUDA IPC, copy engines over NVLink) while the next piece is computed; "
                          "a one-element NCCL all-reduce ends the step") if world > 1 else "none"}


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def stop(self, t0: float, t1: float):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.kill()
        inside = [r for t, r in self.rows if t0 <= t <= t1] or [r for _, r in self.rows[-3:]]
        sm = sorted(float(r[0]) for r in inside if r[0].replace(".", "").isdigit())
        reasons = set()
        for r in inside:
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_max_mhz": float(inside[0][1]) if inside else None,
                "power_w_max": max((float(r[2]) for r in inside), default=None),
                "samples": len(inside), "reasons": sorted(reasons)}


def cpu_reference_run(codes, offsets, lens, n, threads, row_begin=0):
    """Times the reference's own CPU path (oracle/_ref) on rows [row_begin, n) of the triangle."""
    from famsa_b200 import seqio
    from oracle import pyoracle
    letters = []
    for i in range(n):
        o = int(offsets[i])
        letters.append(seqio.decode(codes[o:o + int(lens[i])]))
    rs = pyoracle.RefSeqSet(letters)
    sec, pairs, _ = rs.triangle_mt(row_begin, n, threads, 2)
    rs.close()
    return sec, pairs


# ---------------------------------------------------------------------------------------------- HP-2 leg
DP_MERGES, DP_CARD, DP_WIDTH, DP_SEED = 296, (24, 64), (380, 520), 11
DP_GAPS = (-14850, -1250, -660, -660)            # CParams defaults x1000 (src/core/params.cpp:26-29)


def dp_workload(rank: int):
    """A batch of independent profile-profile merges of the size the upper levels of a 10k x 400 aa guide tree
    produce: 296 (= 2 x 148 SMs) pairs of aligned blocks, 24-64 sequences x 380-520 columns each.  The tables
    are built on the host by famsa_b200.profiles (mirror of CProfile::CalculateCounters/Scores)."""
    from famsa_b200 import profiles
    rng = np.random.default_rng(DP_SEED + rank)
    sm = profiles.synth_score_matrix(rng)
    rows, jobs = [], []
    for _ in range(DP_MERGES):
        pair = []
        for _ in range(2):
            r = profiles.synth_alignment(int(rng.integers(*DP_CARD)), int(rng.integers(*DP_WIDTH)), rng)
            pair.append(r)
        rows.append(pair)
        a = profiles.tables_from_rows(pair[0], sm, DP_GAPS)
        b = profiles.tables_from_rows(pair[1], sm, DP_GAPS)
        jobs.append((a[0], a[1], a[2], b[0], b[1], b[2]))
    return rows, jobs


def dp_cpu_reference(rows, threads, min_seconds=2.0):
    """The reference's CProfile::Align (+ ConstructProfile, inseparable without patching it) over the same
    aligned blocks, one merge per task on `threads` host threads (ComputeAlignment's shape, msa.cpp:375-426).
    The batch is repeated (profiles rebuilt outside the timed calls) until at least min_seconds have been timed."""
    from famsa_b200 import seqio
    from oracle import pyoracle
    dp = pyoracle.RefDp(0)
    dp.set_gaps(DP_GAPS)
    to_str = lambda r: ["".join("-" if c < 0 else seqio.ALPHABET[c] for c in row) + "A" for row in r]
    sec = 0.0
    cells = 0
    while sec < min_seconds:
        p1 = [dp.profile(to_str(a), list(range(len(a)))) for a, _ in rows]
        p2 = [dp.profile(to_str(b), list(range(1000, 1000 + len(b)))) for _, b in rows]
        s1, c1 = dp.align_pairs_mt(p1, p2, threads)
        sec += s1
        cells += c1
    dp.close()
    return sec, cells


def dp_verify_batch(eng, rows, n_paths=48):
    """Untimed: the bench's DP batch against the reference.  The reference builds its CProfile objects from the same
    aligned blocks (dp_cpu_reference's inputs); their score / counter tables go through famsa_dp_align_batch and every
    merge's total score -- and the whole traceback path of the first n_paths merges -- must equal CProfile::Align's."""
    from famsa_b200 import seqio
    from oracle import pyoracle
    dp = pyoracle.RefDp(0)
    dp.set_gaps(DP_GAPS)
    to_str = lambda r: ["".join("-" if c < 0 else seqio.ALPHABET[c] for c in row) + "A" for row in r]
    jobs, profs = [], []
    for a, b in rows:
        na, nb = list(range(len(a))), list(range(1000, 1000 + len(b)))
        p1, p2 = dp.profile(to_str(a), na), dp.profile(to_str(b), nb)
        jobs.append(dp.tables(p1) + dp.tables(p2))
        profs.append((p1, p2, set(na), set(nb)))
    got = eng.dp_align_batch(jobs, np.array(DP_GAPS, dtype=np.int64))
    ok_tot = ok_path = 0
    for k, (p1, p2, na, nb) in enumerate(profs):
        m, total = dp.align(p1, p2, 1)
        ok_tot += int(total == got[k]["total"])
        if k < n_paths:
            # whole traceback path against the C restatement of CProfile::Align (oracle/dp_oracle.c, itself pinned to the
            # reference's goldens and to the live reference by tests/test_oracle_dp.py) on the reference's own tables
            want = pyoracle.dp_align(*jobs[k], np.array(DP_GAPS, dtype=np.int64))
            ok_path += int(want["total"] == total and want["swapped"] == got[k]["swapped"] and np.array_equal(want["path"], got[k]["path"]))
        dp.free(m)
    dp.close()
    return {"totals_equal_to_reference": ok_tot, "of": len(rows), "paths_equal_to_pinned_oracle": ok_path, "paths_checked": min(n_paths, len(rows))}


def bench_dp(eng, torch, dist, world, rank, steps, warmup, l2_flush, stream, want_cpu, dump=None):
    import ctypes as C
    from famsa_b200.binding import DpJob, DpProfile
    rows, jobs = dp_workload(rank)
    n = len(jobs)
    cells = sum((j[0].shape[0] - 1) * (j[3].shape[0] - 1) for j in jobs)
    gaps = np.array(DP_GAPS, dtype=np.int64)
    # device-resident copies of every table
    sc = torch.from_numpy(np.concatenate([np.concatenate([j[0].ravel(), j[3].ravel()]) for j in jobs])).cuda()
    cn = torch.from_numpy(np.concatenate([np.concatenate([j[1].ravel(), j[4].ravel()]) for j in jobs])).cuda()
    arr = (DpJob * n)()
    so = co = 0
    path_total = 0
    for k, j in enumerate(jobs):
        w1, w2 = j[0].shape[0] - 1, j[3].shape[0] - 1
        arr[k].p1 = DpProfile(sc.data_ptr() + 8 * so, cn.data_ptr() + 4 * co, w1, j[2])
        so += (w1 + 1) * 32; co += (w1 + 1) * 32
        arr[k].p2 = DpProfile(sc.data_ptr() + 8 * so, cn.data_ptr() + 4 * co, w2, j[5])
        so += (w2 + 1) * 32; co += (w2 + 1) * 32
        path_total += w1 + w2
    d_res = torch.empty(n * 64, dtype=torch.uint8, device="cuda")
    d_path = torch.empty(path_total, dtype=torch.uint8, device="cuda")

    def step_device():
        eng.dp_align_batch_device(arr, n, gaps, d_res.data_ptr(), d_path.data_ptr(), 0, stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(warmup):
        step_device()
    barrier()
    l0 = eng.kernel_launches()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for s in range(steps):
        l2_flush.fill_(s)
        ev[s][0].record()
        step_device()
        ev[s][1].record()
    barrier()
    launches = eng.kernel_launches() - l0
    if dump is not None:                         # untimed: what the last timed step returned (DpResult records + paths)
        res = d_res.cpu().numpy()
        rec = res.view(np.int64).reshape(-1, 8)[:n]
        poff, plen = res.view(np.uint64).reshape(-1, 8)[:n, 4], res.view(np.uint32).reshape(-1, 16)[:n, 12]
        path = d_path.cpu().numpy()
        dump["dp_total"] = rec[:, 0].astype(np.float64)
        dump["dp_path"] = np.concatenate([path[int(o):int(o) + int(ln)] for o, ln in zip(poff, plen)]).astype(np.float32)
    dev_ms = sum(a.elapsed_time(b) for a, b in ev)
    t = torch.tensor([dev_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms = float(t.item())
    # kernel-only time (prep + T + fill) from the library's own events on the context stream
    eng.dp_align_batch_device(arr, n, gaps, d_res.data_ptr(), d_path.data_ptr(), 0, 0)
    kern_ms = eng.dp_last_timing()[1]
    # e2e through the host-buffer C ABI (job array prebuilt: the timed call is what a C caller makes)
    from famsa_b200.binding import DpResult, ProfMerge
    harr, hkeep, hpath_total = eng.dp_jobs(jobs)
    hres = (DpResult * n)()
    hpath = np.zeros(hpath_total, dtype=np.uint8)
    for _ in range(max(1, warmup // 2)):
        eng.dp_align_batch_raw(harr, n, gaps, hres, hpath)
    barrier()
    t0 = time.time()
    for _ in range(steps):
        eng.dp_align_batch_raw(harr, n, gaps, hres, hpath)
    barrier()
    e2e_s = time.time() - t0
    t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_s = float(t.item())
    h2d = int(sum(j[0].nbytes + j[1].nbytes + j[3].nbytes + j[4].nbytes for j in jobs))
    d2h = int(path_total + 64 * n)
    # e2e with resident profiles (famsa_prof_merge_batch): the children are outputs of the previous tree level and
    # already live in HBM (here: re-uploaded outside the timed region before each step, since a merge consumes
    # them); the timed call aligns, tracebacks, builds the merged tables on the device and returns the paths.
    profs = [p for j in jobs for p in ((j[0], j[1], j[2]), (j[3], j[4], j[5]))]
    res_s = 0.0
    marr = (ProfMerge * n)()
    mids = np.zeros(n, dtype=np.uint32)
    for s in range(steps + 1):
        ids = eng.prof_put(profs)
        for k in range(n):
            marr[k] = ProfMerge(ids[2 * k], ids[2 * k + 1])
        barrier()
        t0 = time.time()
        eng.prof_merge_batch_raw(marr, n, gaps, mids, hres, hpath)
        torch.cuda.synchronize()
        if s:                                    # first pass warms the allocator
            res_s += time.time() - t0
        eng.prof_drop(mids)
    t = torch.tensor([res_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    res_s = float(t.item())
    construct_ms = eng.prof_last_timing()[1]
    out = None
    if rank == 0:
        peak, peak_src = peaks()
        # SURVEY 8(d): per merge (W1+1)(W2+1) direction bytes + traceback + tables + path
        alg = sum((j[0].shape[0]) * (j[3].shape[0]) + 2 * (j[0].shape[0] + j[3].shape[0] - 2)
                  + 160 * j[0].shape[0] + 384 * j[3].shape[0] for j in jobs)
        achieved = alg / (kern_ms / 1e3) / 1e9
        tprof = os.path.join(ROOT, "profiles", "dp_fill_traffic.json")
        dp_traffic = json.load(open(tprof)).get("dram_bytes_per_launch") if os.path.exists(tprof) else None
        out = {"metric": "profile DP cells/sec", "unit": "cells/s", "value": cells * world * steps / (dev_ms / 1e3),
               "ms_per_step": dev_ms / steps,
               "config": {"workload": f"{n} independent profile-profile merges per GPU, {DP_CARD[0]}-{DP_CARD[1]} sequences x "
                                      f"{DP_WIDTH[0]}-{DP_WIDTH[1]} columns each (seed {DP_SEED}), unbanded AlignProfProf + traceback",
                          "cells_per_step_per_gpu": cells, "multi_gpu": "merges sharded across ranks, no collective (replicas per merge)"},
               "e2e": {"value": cells * world * steps / res_s, "unit": "cells/s", "ms_per_step": 1e3 * res_s / steps,
                       "h2d_bytes_per_step": 8 * n, "d2h_bytes_per_step": d2h, "construct_kernel_ms": construct_ms,
                       "note": "famsa_prof_merge_batch, the path INTEGRATION.md wires into ComputeAlignment: child profiles "
                               "resident in HBM (outputs of the previous level), merged tables built on the device "
                               "(ConstructProfile's share, which the CPU baseline also contains), only results + paths return"},
               "e2e_host_tables": {"value": cells * world * steps / e2e_s, "unit": "cells/s", "h2d_bytes_per_step": h2d,
                                   "d2h_bytes_per_step": d2h, "ms_per_step": 1e3 * e2e_s / steps,
                                   "note": "compatibility entry famsa_dp_align_batch: both children's tables cross PCIe on "
                                           "every call (bound by the H2D copy and the host-side packing, does not scale with "
                                           "ranks sharing one host); kept for callers that hold profiles on the host"},
               "gpu_launches": int(launches),
               "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                            "traffic": dp_traffic, "peak_source": peak_src, "kernel": "fb::k_dp_prep + k_dp_fill_compact<NW> + k_dp_trace",
                            "kernel_ms": kern_ms, "algorithmic_bytes": alg,
                            "note": "achieved = SURVEY 8d algorithmic bytes / time of the DP kernels of one batch; traffic = DRAM "
                                    "bytes of the same kernels from ncu (profiles/dp_fill_traffic.json): the column-pair scores T "
                                    "are built in shared memory (IMMA) and never reach HBM; the int64 recurrence is bound by "
                                    "dependent-issue latency, not by HBM: see DESIGN.md section 4"}}
        out["verified_vs_reference"] = None
        if want_cpu:
            from oracle import pyoracle
            if pyoracle.have_ref():
                threads = usable_cpus()
                sec, c = dp_cpu_reference(rows, threads)
                out["cpu_baseline"] = {"value": c / sec, "unit": "cells/s", "cores": threads, "kind": "reference",
                                       "sample": f"the same {n} merges repeated for {sec:.2f} s, CProfile::Align incl. ConstructProfile, one merge per thread task"}
                out["verified_vs_reference"] = dp_verify_batch(eng, rows)
    return out


# ---------------------------------------------------------------------------------------------- C3 / C5 legs
C3_N, C3_SEED = 100000, 2
C5_N, C5_LEN, C5_SEEDS, C5_SEED = 3000000, 250, 100, 3


def bench_c3(eng, torch, dist, world, rank, stream, l2_flush, steps):
    """BASELINE config 3 (strong scaling): the LCS triangle of 100 000 x 400 aa (4 999 950 000 pairs) sharded over the
    ranks, the exchange overlapped piece by piece; every rank ends with the full 10 GB packed triangle."""
    from famsa_b200 import seqio
    codes, offsets, lens = seqio.synth_family(C3_N, LEN, C3_SEED)
    n = len(lens)
    eng.upload(codes, offsets, lens)
    pt = PeerTriangle(eng, n, 2, rank, world, dist)
    full = pt.tensor(torch)
    flag = torch.zeros(1, dtype=torch.int32, device="cuda")

    def step():
        pt.step(torch, stream, 8, flag)

    step()
    dist.barrier(); torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for s in range(steps):
        l2_flush.fill_(s)
        ev[s][0].record(); step(); ev[s][1].record()
    dist.barrier(); torch.cuda.synchronize()
    t = torch.tensor([sum(a.elapsed_time(b) for a, b in ev)], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item()) / steps
    # untimed checks: identical on every rank; oracle spot check on rank 0
    chk = full.to(torch.int64).sum().reshape(1)
    lo, hi = chk.clone(), chk.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN); dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    spot = None
    if rank == 0:
        from oracle import pyoracle
        rng = np.random.default_rng(5)
        spot = True
        for ref in rng.integers(1, n, size=3):
            cols = rng.integers(0, ref, size=200)
            want = pyoracle.lcs_rows(codes, offsets, lens, [int(ref)], cols)[0]
            got = full[tri(int(ref)) + torch.from_numpy(cols).cuda()].cpu().numpy().astype(np.uint32)
            spot = spot and bool(np.array_equal(got, want))
    upgma = None
    if rank == 0:
        try:
            t0 = time.time()
            tree = eng.upgma(0, False, full.data_ptr(), 2)
            upgma = {"ms": 1e3 * (time.time() - t0), "merges": int(len(tree)),
                     "note": "UPGMA on the gathered triangle (famsa_lcs_upgma_from_triangle) on rank 0: float distances + agglomeration on the device"}
        except Exception as e:
            upgma = {"error": str(e)}
    dist.barrier()
    out = {"metric": METRIC, "unit": UNIT, "scaling": "strong", "value": tri(n) / (ms / 1e3), "ms_per_step": ms, "steps": steps, "warmup": 1,
           "upgma_tree": upgma,
           "config": {"workload": f"LCS triangle, {n} x {LEN} aa synthetic family (seed {C3_SEED}), rows sharded over {world} GPUs, "
                                  "every rank's rows computed in 8 pieces, each finished piece copied into every peer's full triangle "
                                  "(CUDA IPC, copy engines over NVLink) while the next is computed", "pairs_per_step": tri(n)},
           "gathered_triangle_identical_on_all_ranks": bool(lo.item() == hi.item()), "oracle_spot_check": spot}
    del full
    pt.close(torch)
    torch.cuda.empty_cache()
    return out


def c5_family(torch, n, L, seed):
    """3M ABC-transporter-like sequences x 250 aa (SURVEY 8d: 2-level family, 300 sub-roots at 0.25 from the root, members
    at 0.20 from their sub-root), generated on the GPU because a host generator would take minutes; lengths L-7 .. L."""
    g = torch.Generator(device="cuda"); g.manual_seed(seed)
    root = torch.randint(0, 20, (L,), generator=g, device="cuda", dtype=torch.int8)
    subs = root.repeat(300, 1)
    m = torch.rand((300, L), generator=g, device="cuda") < 0.25
    subs[m] = torch.randint(0, 20, (int(m.sum()),), generator=g, device="cuda", dtype=torch.int8)
    which = torch.randint(0, 300, (n,), generator=g, device="cuda")
    codes = subs[which]
    chunk = 1 << 18
    for a in range(0, n, chunk):
        blk = codes[a:a + chunk]
        m = torch.rand(blk.shape, generator=g, device="cuda") < 0.20
        blk[m] = torch.randint(0, 20, (int(m.sum()),), generator=g, device="cuda", dtype=torch.int8)
    lens = (L - torch.randint(0, 8, (n,), generator=g, device="cuda")).to(torch.int32)
    order = torch.argsort(lens, descending=True, stable=True)       # FAMSA's own order: longest first
    codes, lens = codes[order].contiguous(), lens[order]
    offsets = (torch.arange(n, device="cuda", dtype=torch.int64) * L)
    return codes.cpu().numpy().reshape(-1), offsets.cpu().numpy().astype(np.uint64), lens.cpu().numpy().astype(np.uint32)


def bench_c5(eng, torch, dist, world, rank, stream, steps, dump=None):
    """BASELINE config 5, the LCS side of -medoidtree: the assignment step of FastTree<>::makeEvaluation (FastTree.cpp:
    309-324) for 100 seeds x 3 000 000 sequences x 250 aa, the sequences sharded over the ranks, one NCCL MIN all-reduce of
    the packed (distance, seed) pairs."""
    from famsa_b200.binding import unpack_assignment
    codes, offsets, lens = c5_family(torch, C5_N, C5_LEN, C5_SEED)
    n = len(lens)
    eng.upload(codes, offsets, lens)
    seeds = np.random.default_rng(C5_SEED).choice(n, size=C5_SEEDS, replace=False).astype(np.uint32)
    packed = torch.empty(n, dtype=torch.int64, device="cuda")

    def shard_fn(r, w, t):
        eng.assign_shard(seeds, r, w, t.data_ptr(), 0, stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    assign_allreduce(shard_fn, packed, rank, world, dist)
    barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for s in range(steps):
        ev[s][0].record(); assign_allreduce(shard_fn, packed, rank, world, dist); ev[s][1].record()
    barrier()
    t = torch.tensor([sum(a.elapsed_time(b) for a, b in ev)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item()) / steps
    out = None
    if rank == 0:
        a, d = unpack_assignment(packed.cpu().numpy())
        if dump is not None:
            dump["c5_assignment"] = a.astype(np.float32)
            dump["c5_min_dist"] = d
        same = None
        if world > 1:                                # untimed: the unsharded call on this rank gives the same answer
            a1, d1 = eng.assign(seeds, 0)
            same = bool(np.array_equal(a, a1) and np.array_equal(d, d1))
        pairs = n * C5_SEEDS
        peak, _ = peaks()
        b_pair = float(lens.mean()) + 4.0
        out = {"metric": METRIC, "unit": UNIT, "scaling": "strong", "value": pairs / (ms / 1e3), "ms_per_step": ms, "steps": steps,
               "config": {"workload": f"medoid assignment: {C5_SEEDS} seed rows x {n} sequences x {C5_LEN} aa (2-level synthetic family, "
                                      f"seed {C5_SEED}), sequences sharded over {world} GPU(s), one MIN all-reduce of 8 B per sequence",
                          "pairs_per_step": pairs},
               "roofline": {"bound": "hbm", "achieved": pairs * b_pair / (ms / 1e3) / 1e9 / world, "peak": peak, "unit": "GB/s",
                            "frac": pairs * b_pair / (ms / 1e3) / 1e9 / world / peak, "bytes_per_pair": b_pair,
                            "note": "per GPU, whole step (seed-row tiles + gather + arg-min + all-reduce) against the HBM contract roofline"},
               "assigned_to_seed0": int((a == 0).sum()), "cost": float(np.add.accumulate(d.astype(np.float32))[-1]),
               "identical_to_unsharded": same}
    del packed
    torch.cuda.empty_cache()
    return out


# ---------------------------------------------------------------------------------------------- whole-tree DP leg
TREE_SYNTH = (2000, 400, 17, 1)          # sequences, length, family seed, tree seed


def tree_workloads():
    """BASELINE config 4 (test/hemopexin, every merge of the golden medoid-sl tree and of the default -gt sl tree; the
    fixtures carry the reference's per-merge totals and path checksums) and a synthetic 2000 x 400 aa family under a
    random guide tree.  Returns [(name, sequences, merges (n-1, 2), gaps, fixture or None)]."""
    from famsa_b200 import seqio
    G = os.path.join(ROOT, "tests", "golden")
    out = []
    for f in ("hemopexin_medoid_sl", "hemopexin_sl"):
        z = np.load(os.path.join(G, f + ".npz"))
        out.append((f, [str(x) for x in z["seqs"]], np.asarray(z["merges"], dtype=np.int32), np.asarray(z["gaps"], dtype=np.int64), z))
    n, L, seed, tseed = TREE_SYNTH
    codes, off, lens = seqio.synth_family(n, L, seed, sort_desc=False)
    seqs = [seqio.decode(codes[int(o):int(o) + int(l)]) for o, l in zip(off, lens)]
    rng = np.random.default_rng(tseed)
    alive, merges = list(range(n)), []
    while len(alive) > 1:                # random binary merge order, 5 % chain-like steps (tests/dp_cases.random_tree)
        if rng.random() < 0.05 and merges:
            a = alive.pop(); b = alive.pop(int(rng.integers(len(alive))))
        else:
            a = alive.pop(int(rng.integers(len(alive)))); b = alive.pop(int(rng.integers(len(alive))))
        merges.append((a, b)); alive.append(n + len(merges) - 1)
    out.append((f"synthetic {n} x {L} aa family, random guide tree", seqs, np.asarray(merges, dtype=np.int32), out[0][3], None))
    return out


def bench_dp_tree(eng, torch, dist, world, rank, steps, want_cpu, dump=None):
    """Whole progressive alignments through famsa_prof_align_tree (one call per tree: every merge of the guide tree,
    profiles resident in HBM, per-merge records + paths back on the host), timed by the host clock around the call
    plus the path fetch.  Next to it the reference's own ComputeAlignment loop (CProfileQueue + worker threads) on all
    host cores, repeated for >= 2 s."""
    import zlib
    from famsa_b200 import seqio
    sm = np.load(os.path.join(ROOT, "tests", "golden", "adeno_upgma_merges.npz"))["score_matrix"]
    legs = []
    for name, seqs, merges, gaps, fx in tree_workloads():
        codes, off, lens = seqio.pack([seqio.encode(x) for x in seqs])
        eng.upload(codes, off, lens)
        eng.prof_set_scoring(sm)
        root, res, st = eng.align_tree(merges, gaps)          # warm-up + the run that is verified
        eng.prof_drop([root])
        check = None
        if fx is not None:
            check = bool([r["total"] for r in res] == [int(t) for t in fx["totals"]]
                         and [zlib.crc32(r["path"].tobytes()) for r in res] == [int(c) for c in fx["path_crc"]])
        l0 = eng.kernel_launches()
        walls, devs = [], []
        raw = eng.align_tree_buffers(merges, gaps, st)       # the arrays a C caller passes: built once
        for _ in range(steps):
            if world > 1:
                dist.barrier()
            t0 = time.time()
            root, st = eng.align_tree_raw(raw)                # famsa_prof_align_tree + famsa_prof_tree_paths
            walls.append(time.time() - t0)
            devs.append(st["device_ms"])
            eng.prof_drop([root])
        launches = eng.kernel_launches() - l0
        if dump is not None:                      # what the last timed call returned: per-merge totals and paths
            recs = raw["res"][:raw["n"]]
            key = f"dp_tree{len(legs)}"
            dump[key + "_total"] = np.array([r.total_score for r in recs], dtype=np.float64)
            dump[key + "_path"] = np.concatenate([raw["path"][r.path_offset:r.path_offset + r.path_len] for r in recs]).astype(np.float32)
        wall = sorted(walls)[len(walls) // 2]
        t = torch.tensor([wall], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        wall = float(t.item())
        leg = {"tree": name, "n_seqs": len(seqs), "merges": int(len(merges)), "cells": int(st["cells"]), "final_width": int(len(res[-1]["path"])),
               "wall_ms": 1e3 * wall, "device_ms": sorted(devs)[len(devs) // 2], "cells_per_s": st["cells"] * world / wall,
               "batches": int(st["n_batches"]), "max_batches_in_flight": int(st["max_in_flight"]),
               "gpu_launches_per_tree": int(launches // max(1, steps)),
               "identical_to_reference_fixture": check}
        if want_cpu and rank == 0:
            from oracle import pyoracle
            if pyoracle.have_ref():
                threads = usable_cpus()
                dp = pyoracle.RefDp(len(seqs))
                dp.set_gaps(gaps)
                sec, reps, rows, total = 0.0, 0, None, None
                while sec < 2.0:
                    out = dp.align_tree_mt(seqs, merges, threads, want_rows=(reps == 0))
                    sec += out[0]; reps += 1
                    if len(out) > 4:
                        rows, total = out[4], out[2]
                dp.close()
                leg["cpu_reference"] = {"wall_ms": 1e3 * sec / reps, "cores": threads, "repeats": reps,
                                        "what": "the reference's ComputeAlignment loop (CProfileQueue + workers, msa.cpp:360-438) on the same tree"}
                leg["speedup_vs_reference"] = (sec / reps) / wall
                # untimed: the alignment assembled from the GPU's paths is the reference's alignment, row for row
                sys.path.insert(0, os.path.join(ROOT, "tests"))
                from dp_cases import assemble_rows
                mine = assemble_rows(seqs, [tuple(int(x) for x in m) for m in merges], res)
                leg["alignment_identical_to_reference"] = bool(mine == rows and res[-1]["total"] == total)
        legs.append(leg)
    return legs


def usable_cpus() -> int:
    """Host threads this process may really use: min(affinity, cgroup cpu quota)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(int(q) / int(p))))
    except (OSError, ValueError):
        pass
    return n


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import pyoracle
    (codes, offsets, lens), n = workload(args.gpus)
    threads = usable_cpus()
    if not pyoracle.have_ref():
        emit({"impl": "reference", "unavailable": "oracle/_ref/libfamsa_ref.so not built"})
        return
    # bounded sample: the last rows of the triangle holding ~1/4 of the pairs when the set is large
    row_begin = 0 if n <= 12000 else int(n * math.sqrt(0.75))
    for _ in range(args.warmup):
        cpu_reference_run(codes, offsets, lens, n, threads, max(row_begin, n - 800))
    secs, pairs = 0.0, 0
    for _ in range(args.steps):
        s, p = cpu_reference_run(codes, offsets, lens, n, threads, row_begin)
        secs += s
        pairs = p
    value = pairs * args.steps / secs
    sample = f"triangle rows [{row_begin},{n}) of {n} x {LEN} aa = {pairs} pairs/step"
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64",
            "data": "synthetic", "config": config_for(n, args.gpus),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "reference",
                             "sample": sample + "; CLCSBP AVX2 via calculateDistanceVector, one row per task"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    rows, _ = dp_workload(0)
    sec, cells = dp_cpu_reference(rows, threads)
    line["dp"] = {"metric": "profile DP cells/sec", "unit": "cells/s", "value": cells / sec, "cores": threads,
                  "sample": f"{len(rows)} merges of the b200 arm's DP workload, CProfile::Align incl. ConstructProfile ({sec:.2f} s)"}
    emit(line)


DUMP_SAMPLE, DUMP_SEED, DUMP_LIMIT = 1 << 20, 12345, 64 << 20


def dump_triangle(torch, tri_dev, total_pairs, dump):
    """The packed uint16 LCS triangle of the last timed step: a fixed, seeded sample of DUMP_SAMPLE pairs (sorted
    packed indices) and the sum over every pair."""
    idx = np.sort(np.random.default_rng(DUMP_SEED).choice(total_pairs, size=min(DUMP_SAMPLE, total_pairs), replace=False))
    t = tri_dev.view(torch.int16)[:total_pairs].to(torch.int32) & 0xFFFF
    dump["lcs_triangle_index"] = idx.astype(np.float64)
    dump["lcs_triangle_sample"] = t[torch.from_numpy(idx).cuda()].cpu().numpy().astype(np.float32)
    dump["lcs_triangle_sum"] = np.array([t.to(torch.int64).sum().item()], dtype=np.float64)


def write_dump(out_dir: str, dump: dict) -> dict:
    """Writes every array as out_dir/<name>.npy; returns {name: shape} for the JSON line."""
    total = sum(a.nbytes for a in dump.values())
    if total > DUMP_LIMIT:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in dump.items():
        assert a.dtype in (np.float32, np.float64), name
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return {"dir": out_dir, "bytes": int(total), "arrays": {k: list(a.shape) for k, a in dump.items()}}


_REAL_STDOUT = None


def emit(line: dict):
    """The one JSON line goes to the real stdout; everything else any library prints (NCCL's version banner,
    warnings) was redirected to stderr at start-up."""
    data = (json.dumps(line) + "\n").encode()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, data)


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the timed legs computed in their last step as DIR/<name>.npy (float32 / float64)")
    args = ap.parse_args()
    if args.steps < 1:
        raise SystemExit("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist
    import famsa_b200

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    (codes, offsets, lens), n = workload(world)
    dump = {} if args.dump_outputs and rank == 0 else None
    bounds = row_shards(n, world)
    rb, re = bounds[rank], bounds[rank + 1]
    my_pairs = tri(re) - tri(rb)
    total_pairs = tri(n)
    max_shard = max(shard_sizes(bounds))

    eng = famsa_b200.Engine(local)
    eng.upload(codes, offsets, lens)                       # resident inputs for the `value` leg
    d_block = torch.empty(max(max_shard, 1), dtype=torch.int16, device="cuda")
    pt = PeerTriangle(eng, n, 2, rank, world, dist) if world > 1 else None   # every rank's full packed triangle, mapped by its peers
    d_full = pt.tensor(torch) if pt else None
    flag = torch.zeros(1, dtype=torch.int32, device="cuda")
    side = torch.cuda.Stream()                             # non-default stream shared by our kernels and NCCL
    torch.cuda.set_stream(side)
    stream = side.cuda_stream
    l2_flush = torch.empty(192 * 1024 * 1024, dtype=torch.uint8, device="cuda")

    def step_device():
        if world == 1:
            eng.triangle_device(rb, re, d_block.data_ptr(), 2, stream)
        else:
            pt.step(torch, stream, 8, flag)                # own rows in 8 pieces + peer copies, then a one-element all-reduce

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- value: device-resident
    for _ in range(args.warmup):
        step_device()
    barrier()
    launches0 = eng.kernel_launches()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    wall0 = time.time()
    for s in range(args.steps):
        l2_flush.fill_(s)                                  # L2 flush between timed iterations (untimed)
        ev[s][0].record()
        step_device()
        ev[s][1].record()
    barrier()
    wall1 = time.time()
    launches = eng.kernel_launches() - launches0
    if dump is not None:
        dump_triangle(torch, d_block if world == 1 else d_full, total_pairs, dump)
    dev_ms = sum(a.elapsed_time(b) for a, b in ev)
    t = torch.tensor([dev_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms = float(t.item())
    clocks = sampler.stop(wall0, wall1) if rank == 0 else None
    value = total_pairs * args.steps / (dev_ms / 1e3)

    # the same steps without the exchange: what the all-gather still costs after overlapping
    exchange = None
    if world > 1:
        evc = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        barrier()
        for s in range(args.steps):
            l2_flush.fill_(s)
            evc[s][0].record()
            eng.triangle_device(rb, re, d_block.data_ptr(), 2, stream)
            evc[s][1].record()
        barrier()
        t = torch.tensor([sum(a.elapsed_time(b) for a, b in evc)], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        comp_ms = float(t.item())
        # every rank must hold the same gathered triangle: compare a checksum
        chk = d_full.view(torch.int16).to(torch.int64).sum().reshape(1)
        lo, hi = chk.clone(), chk.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN); dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        whole = torch.empty(total_pairs, dtype=torch.int16, device="cuda")        # untimed: the whole triangle on this GPU alone
        eng.triangle_device(0, n, whole.data_ptr(), 2, stream)
        torch.cuda.synchronize()
        same = torch.tensor([int(torch.equal(whole, d_full))], dtype=torch.int32, device="cuda")
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        del whole
        exchange = {"compute_only_ms_per_step": comp_ms / args.steps, "all_gather_exposed_ms_per_step": (dev_ms - comp_ms) / args.steps,
                    "gathered_bytes_per_rank": int(total_pairs * 2), "gathered_triangle_identical_on_all_ranks": bool(lo.item() == hi.item()),
                    "gathered_triangle_equals_single_gpu_triangle_on_every_rank": bool(same.item() == 1)}

    # dominant kernel, timed live with CUDA events on its launch stream (single launch class at this config)
    kern_ms = []
    for _ in range(3):
        l2_flush.fill_(1)
        eng.triangle_device(rb, re, d_block.data_ptr(), 2, 0)   # ctx stream: synchronises + records timing
        kern_ms.append(eng.last_timing()[1])
    kern_ms = sorted(kern_ms)[1]

    # ---------------- e2e: host buffers through the C ABI, copies inside the timed region
    h_out = torch.empty(max(my_pairs, 1), dtype=torch.int16).pin_memory()
    h_np = h_out.numpy().view(np.uint16)
    codes_p = torch.from_numpy(codes).pin_memory().numpy()

    def step_e2e():
        # N > 1: every rank's row block returns to its own host process (a row-partitioned consumer, e.g. the rows a
        # distributed tree builder owns); there is no collective on this path
        eng.upload(codes_p, offsets, lens)
        eng.triangle(rb, re, out=h_np)

    for _ in range(max(1, args.warmup // 2)):
        step_e2e()
    barrier()
    t0 = time.time()
    for _ in range(args.steps):
        step_e2e()
    barrier()
    e2e_s = time.time() - t0
    t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_s = float(t.item())
    e2e_value = total_pairs * args.steps / e2e_s
    h2d = int(codes.nbytes + offsets.nbytes + lens.nbytes)
    d2h = int(my_pairs * 2)

    if rank == 0:
        peak, peak_src = peaks()
        mean_len = float(lens.mean())
        b_pair = mean_len + 4.0                           # SURVEY 8(d): streamed residues (u8) + u32 result
        achieved = my_pairs * b_pair / (kern_ms / 1e3) / 1e9
        prof = os.path.join(ROOT, "profiles", "lcs_tile_traffic.json")
        traffic = json.load(open(prof)).get("dram_bytes_per_launch") if os.path.exists(prof) else None
        word_steps = my_pairs * mean_len * math.ceil(mean_len / 32)        # 32-bit limb updates
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": config_for(n, world), "rows_of_rank0": [rb, re],
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": 1e3 * e2e_s / args.steps,
                    "note": ("per rank: upload + own row block + D2H of that block to the rank's own host consumer; byte counts are per rank"
                             if world > 1 else "famsa_lcs_upload + famsa_lcs_triangle with host buffers")},
            "exchange": exchange,
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "peak_source": peak_src, "kernel": "fb::k_lcs_tile<NL>",
                         "kernel_ms": kern_ms, "bytes_per_pair": b_pair,
                         "note": "integer-ALU bound, not HBM bound: see alu_model"},
            "alu_model": {"limb_steps_per_s": word_steps / (kern_ms / 1e3),
                          "int_ops_per_limb_step": 3,
                          "alu_pipe_peak_lane_ops_per_s": 148 * 64 * (clocks["sm_mhz"] or 0) * 1e6 if clocks else None},
        }
        if clocks and clocks.get("sm_mhz"):
            line["alu_model"]["frac_of_alu_pipe"] = (3 * word_steps / (kern_ms / 1e3)) / (148 * 64 * clocks["sm_mhz"] * 1e6)
        if world == 1 and not args.no_cpu_baseline:
            from oracle import pyoracle
            if pyoracle.have_ref():
                threads = usable_cpus()
                sec, pairs = cpu_reference_run(codes, offsets, lens, n, threads, 0)
                line["cpu_baseline"] = {"value": pairs / sec, "unit": UNIT, "cores": threads, "kind": "reference",
                                        "sample": f"whole {n} x {LEN} aa triangle ({pairs} pairs, {sec:.2f} s), "
                                                  "oracle/_ref AVX2 path, one row per task"}
            else:
                n_s = 600
                t0 = time.time()
                pyoracle.lcs_triangle(codes, offsets, lens, n - n_s, n)
                sec = time.time() - t0
                pairs = tri(n) - tri(n - n_s)
                line["cpu_baseline"] = {"value": pairs / sec, "unit": UNIT, "cores": 1, "kind": "port",
                                        "sample": f"last {n_s} rows ({pairs} pairs)"}
    dp = bench_dp(eng, torch, dist, world, rank, args.steps, args.warmup, l2_flush, stream,
                  want_cpu=(world == 1 and not args.no_cpu_baseline), dump=dump)
    dp_tree = bench_dp_tree(eng, torch, dist, world, rank, args.steps, want_cpu=(world == 1 and not args.no_cpu_baseline), dump=dump)
    if pt:
        d_full = None
        pt.close(torch)
    c3 = bench_c3(eng, torch, dist, world, rank, stream, l2_flush, args.steps) if world > 1 else None
    c5 = bench_c5(eng, torch, dist, world, rank, stream, args.steps, dump=dump)
    if rank == 0:
        line["dp"] = dp
        line["dp_tree"] = dp_tree
        line["c3_triangle_100k"] = c3 if c3 else {"skipped": "strong-scaling leg: runs when launched on more than one GPU"}
        line["c5_medoid_assignment_3m"] = c5
        line["gpu_launches"] = int(launches) + (dp["gpu_launches"] if dp else 0)
        if world == 1:
            # informational: the default guide tree (-gt sl) end to end on the same set -- famsa_lcs_prim =
            # LCS triangle + Transform + MST (Boruvka rounds under MSTPrim's edge order) + Prim-order replay
            try:
                eng.upload(codes, offsets, lens)
                eng.prim(0)
                t0 = time.time()
                ef, _, ed, _ = eng.prim(0)
                wall = time.time() - t0
                tot, lcs_ms, _ = eng.last_timing()
                line["guide_tree_sl"] = {"ms": 1e3 * wall, "device_ms": tot, "lcs_kernels_ms": lcs_ms, "n_seqs": int(n),
                                         "edges": int(len(ef)), "sum_dist": float(ed.sum()),
                                         "note": "MSTPrim<indel075_div_lcs> tree of the bench set through famsa_lcs_prim; "
                                                 "the reference builds it in cpu_baseline's LCS time plus its Prim loop"}
            except Exception as e:                     # never let the extra leg break the contract line
                line["guide_tree_sl"] = {"error": str(e)}
            # informational: the UPGMA guide tree (-gt upgma) end to end -- famsa_lcs_upgma = LCS triangle + float Transform +
            # UPGMA<>::computeTree's agglomeration, all on the device, only the n-1 merges return
            try:
                eng.upgma(0)
                t0 = time.time()
                tree = eng.upgma(0)
                wall = time.time() - t0
                tot, lcs_ms, _ = eng.last_timing()
                line["guide_tree_upgma"] = {"ms": 1e3 * wall, "device_ms": tot, "lcs_kernels_ms": lcs_ms, "n_seqs": int(n), "merges": int(len(tree)),
                                            "checksum": int((tree.astype(np.int64) * np.arange(1, 2 * len(tree) + 1).reshape(-1, 2)).sum()),
                                            "note": "UPGMA<indel075_div_lcs>::run of the bench set through famsa_lcs_upgma (no n^2 D2H)"}
            except Exception as e:
                line["guide_tree_upgma"] = {"error": str(e)}
        if dump is not None:
            line["dump_outputs"] = write_dump(args.dump_outputs, dump)
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
