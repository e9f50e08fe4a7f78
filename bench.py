#!/usr/bin/env python3
"""Benchmark of the kmerseek sketch-and-search hot path on B200 (contract: see the task brief, section 4).

One "step" = one index build of this rank's shard of the workload's proteome, already resident in HBM:
    fused sketch kernel -> sort by hash -> CSR build (ks_index_clear + ks_index_sketch_resident +
    ks_index_finalize through the C ABI).  The library picks the build path from the parameters and the data
    (`config.build_path`: dense k-mer space path for hp with k <= 24; general path with the unstable or the stable
    partition otherwise, DESIGN.md section 3).
`value` = residues/s over all ranks with inputs resident in HBM; `e2e` = the same metric through the public
host API with HOST buffers (pinned 5-bit packed residues + offsets -> H2D -> build -> stats read back) inside the timed
region.

Multi-GPU (`--gpus N` under torchrun): STRONG scaling -- ONE fixed proteome (the workload's, same seed at every N) is
sharded by protein over the ranks (shard.plan_shards); the build has no collective.  The search leg (BASELINE.json
configs[2]: 10 000 planted query domains, dayhoff k=16) runs on an index of the same proteome through
ks_shard_search_batch (NCCL all-gather of counts + grouped send/recv of the shards' result blocks + counting merge on
rank 0) and is checked against a single-GPU search of the unsharded proteome on rank 0.

--impl reference times the CPU restatement of the reference's own algorithm (oracle/, the reference is Rust with
un-vendored crates and cannot be built in this image) on all host cores: the linear-cost variant on the FULL workload
(same config as the GPU arm) and the faithful-cost port (quadratic) on a bounded sample.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json configs[1]: Swiss-Prot-sized index build, hp k=24 scaled=1 (the config the metric is quoted on)
    "c2_swissprot_hp_k24_s1": dict(n_residues=200_000_000, k=24, moltype="hp", scaled=1, seed=20260102),
    # BASELINE.json configs[2]: the proteome of C2 under dayhoff k=16 (the search leg's index)
    "c3_search_dayhoff_k16_s1": dict(n_residues=200_000_000, k=16, moltype="dayhoff", scaled=1, seed=20260102),
    # the north_star target run
    "target_100m_dayhoff_k16_s1": dict(n_residues=100_000_000, k=16, moltype="dayhoff", scaled=1, seed=20260103),
    "c4_slice_protein_k7_s10": dict(n_residues=1_000_000_000, k=7, moltype="protein", scaled=10, seed=20260104),
    # BASELINE.json configs[3]: UniRef50-scale, 5 G residues, protein k=7 scaled=10, over 2 / 4 / 8 GPUs.  The proteome is 64
    # blocks of 78.125 M residues (block i: generator seed + i), so that every rank can make its own part without
    # holding 5 GB per process: rank r of N owns blocks [64 r / N, 64 (r + 1) / N).  Build legs only (no search leg).
    "c4_uniref50_protein_k7_s10": dict(n_residues=5_000_000_000, k=7, moltype="protein", scaled=10, seed=20260104, blocks=64),
    "small": dict(n_residues=5_000_000, k=24, moltype="hp", scaled=1, seed=20260102),
}
SEARCH_WORKLOAD = "c3_search_dayhoff_k16_s1"
BUILD_PATHS = {0: "general", 1: "dense k-mer space", 2: "dense k-mer space, library key sort",
               3: "general, unstable partition"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel from the committed `ncu --set full`
# captures of the C2 workload on one GPU (profiles/): only meaningful for that workload at N = 1, null otherwise.
TRAFFIC_C2 = {"dense_bucket_kernel": 1_642_193_000 + 3_709_222_000}  # profiles/r02_s_ncu_full_raw_c2_build.csv
# the same for the per-query kernel of the search leg (10 000 queries against the C3 index, pairs only):
# profiles/r02_s_ncu_full_raw_c3_search.csv -- random 32-byte sector gathers (directory, keys, groups, postings, protein
# sizes), which is why it is more than ten times the algorithmic bytes
TRAFFIC_C3_SEARCH = {"query_kernel": 514_447_000 + 22_040_000}


def sketch_bytes(n_res, n_prot, n_tuples):
    """SURVEY 8(d) / BASELINE.md section 3: read residues + offsets, write (u64 hash, u32 protein, u32 pos)."""
    return n_res + (n_prot + 1) * 8 + n_tuples * 16


def build_bytes(n_tuples, n_unique):
    """SURVEY 8(d): one logical pass -- tuples in, payload + keys + row_ptr out (extra passes are implementation traffic)."""
    return n_tuples * 16 + n_tuples * 8 + n_unique * 8 + (n_unique + 1) * 4


def search_bytes(q_res, q_hashes, hits, pairs):
    """SURVEY 8(d): query in, one key probe + row_ptr pair per query hash, postings + hit rows, 48 B of scores per pair."""
    return q_res + q_hashes * 8 + q_hashes * 16 + hits * 8 + hits * 20 + pairs * 48


# --dump-outputs: rows kept per column.  The dumped tables have at most 43 float64 columns of this length (index and
# target index: hash hi/lo, row start hi/lo, row length hi/lo, posting pid, pos; search: 6 hit and 21 pair columns),
# about 43 MB in all.
DUMP_ROWS = 1 << 17
DUMP_SEED = 20260101


def dump_columns(prefix, cols):
    """One result table (columns of equal length) as {prefix + column: float64 array}: every row when there are at most
    DUMP_ROWS, else the same seeded sample of rows in every column.  A 64-bit integer column becomes its exact 32-bit
    halves `<column>_hi` / `<column>_lo`; every integer column also gets `<column>_sha256`, the digest of the whole
    column as eight 32-bit words, so that the rows outside the sample are compared too."""
    n = len(next(iter(cols.values())))
    rows = None if n <= DUMP_ROWS else np.sort(np.random.default_rng(DUMP_SEED).choice(n, DUMP_ROWS, replace=False))
    out = {}
    for name, a in cols.items():
        a = np.ascontiguousarray(a)
        s = a if rows is None else a[rows]
        if a.dtype.kind in "ui":
            out[prefix + name + "_sha256"] = np.frombuffer(hashlib.sha256(a).digest(), dtype="<u4").astype(np.float64)
            if a.dtype.itemsize == 8:
                s = s.astype(np.uint64)
                out[prefix + name + "_hi"] = (s >> np.uint64(32)).astype(np.float64)
                out[prefix + name + "_lo"] = (s & np.uint64(0xFFFFFFFF)).astype(np.float64)
                continue
        out[prefix + name] = s.astype(np.float64)
    return out


def dump_index(prefix, idx):
    """The finalized index as a caller of ks_index_csr receives it: sorted unique hashes with their posting rows, and
    the postings (protein, position)."""
    keys, row_ptr, pid, pos = idx.csr()
    return {**dump_columns(prefix + "key_", {"hash": keys, "row_start": row_ptr[:-1], "row_len": np.diff(row_ptr)}),
            **dump_columns(prefix + "posting_", {"pid": pid, "pos": pos})}


def write_dump(directory, arrays):
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


_PROTEOME_CACHE = {}


def cpu_baseline_run(cfg, faithful, sample_residues, threads):
    from oracle import oracle as O
    from kmerseek_b200 import synth
    key = (sample_residues, cfg["seed"])
    if key not in _PROTEOME_CACHE:
        _PROTEOME_CACHE.clear()
        _PROTEOME_CACHE[key] = synth.proteome(sample_residues, cfg["seed"])
    res, offs = _PROTEOME_CACHE[key]
    t0 = time.perf_counter()
    n, uniq, kept = O.cpu_baseline(res, offs, cfg["k"], cfg["moltype"], cfg["scaled"], faithful=faithful, n_threads=threads)
    dt = time.perf_counter() - t0
    return n / dt, dt, uniq, kept


def run_reference(args, cfg, wname):
    """The reference arm.  `value`: the CPU restatement of the reference's per-protein algorithm (translate, MurmurHash3,
    FracMinHash filter, sorted mins + abundances, positions per hash) over the FULL workload on all host threads, in
    1000-record batches like src/rust/index.rs:938-941,993-1005, with the reference's two super-linear steps made linear
    (binary-search membership instead of `Vec::contains`, index.rs:769; no sorted-Vec combined insert, :824-827) -- the
    only form of the algorithm that can finish this config (SURVEY F8).  `faithful`: the same port with the reference's
    cost structure kept, on a bounded sample (quadratic: the rate depends on the sample)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    # the whole run must end within a few minutes: size the per-step sample from a short trial (the full workload when
    # the host is fast enough, which makes this arm the same config as the GPU arm)
    trial = min(cfg["n_residues"], 10_000_000)
    rate, _, _, _ = cpu_baseline_run(cfg, False, trial, threads)
    budget_s = 200.0 / max(1, args.warmup + args.steps)
    sample = int(min(cfg["n_residues"], max(trial, rate * budget_s)))
    vals = []
    for i in range(args.warmup + args.steps):
        v, dt, _, _ = cpu_baseline_run(cfg, False, sample, threads)
        if i >= args.warmup:
            vals.append((v, dt))
    v = float(np.mean([x[0] for x in vals]))
    ms = float(np.mean([x[1] for x in vals]) * 1e3)
    fv, fdt, _, _ = cpu_baseline_run(cfg, True, args.reference_sample, threads)
    line = {
        "impl": "reference", "metric": "residues/s sketched+indexed", "value": v, "unit": "residues/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": wname, "k": cfg["k"], "moltype": cfg["moltype"], "scaled": cfg["scaled"],
                   "residues": sample, "same_config_as_gpu_arm": sample == cfg["n_residues"]},
        "cpu_baseline": {"value": v, "unit": "residues/s", "cores": threads, "kind": "port",
                         "sample": (f"the full workload ({sample} residues)" if sample == cfg["n_residues"] else
                                    f"first {sample} of {cfg['n_residues']} residues") +
                                   " per step; linear-cost variant of the reference's algorithm (binary-search membership, no "
                                   "combined-sketch insert)",
                         "faithful": {"value": fv, "unit": "residues/s", "cores": threads,
                                      "sample": f"first {args.reference_sample} residues, reference cost structure kept (two "
                                                f"passes, linear contains, sorted-Vec combined insert: quadratic), {fdt:.1f} s"}},
        "e2e": {"value": v, "unit": "residues/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def run_c5_sweep(args):
    """BASELINE.json configs[4]: k 5..24 x {protein, dayhoff, hp}, scaled 1, 10 M-residue proteome, one GPU.  Per cell: the
    fused sketch kernel's time (CUDA events of the library) and the whole resident build; hit-list equality of all 60
    cells is tests/test_gpu_c5_sweep.py."""
    import torch
    import kmerseek_b200 as K
    from kmerseek_b200 import _ffi, synth
    if int(os.environ.get("RANK", "0")) != 0:
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (kmerseek_b200 has no CPU fallback)")
    L = _ffi.lib()
    chk = K.errors.check
    peak, _ = peaks()
    n_res = 10_000_000
    res, offs = synth.proteome(n_res, 20260105)
    prot = K.Proteome.from_packed(res, offs)
    cells = []
    for moltype in ("protein", "dayhoff", "hp"):
        for k in range(5, 25):
            idx = K.ProteomeIndex("c5", k, 1, moltype)
            chk(L.ks_index_upload(idx._h, prot._h))
            sk, tot = [], []
            for i in range(max(args.warmup, 2) + args.steps):
                t0 = time.perf_counter()
                chk(L.ks_index_clear(idx._h)); chk(L.ks_index_sketch_resident(idx._h)); chk(L.ks_index_finalize(idx._h))
                st = idx.stats()
                if i >= max(args.warmup, 2):
                    tot.append((time.perf_counter() - t0) * 1e3)
                    sk.append(st["ms_sketch"])
            nt, nu = st["n_tuples"], st["n_unique_hashes"]
            b = sketch_bytes(n_res, len(offs) - 1, nt)
            cells.append({"moltype": moltype, "k": k, "ms_sketch": round(float(np.mean(sk)), 4), "ms_build_wall": round(float(np.mean(tot)), 4),
                          "sketch_residues_per_s": n_res / (float(np.mean(sk)) * 1e-3), "sketch_frac_of_hbm": b / float(np.mean(sk)) / 1e6 / peak,
                          "build_residues_per_s": n_res / (float(np.mean(tot)) * 1e-3), "tuples": nt, "unique_hashes": nu,
                          "build_path": BUILD_PATHS[st["build_path"]]})
            idx.close()
    v = float(np.exp(np.mean([np.log(c["sketch_residues_per_s"]) for c in cells])))
    print(json.dumps({"metric": "residues/s sketched (geometric mean over the 60 cells)", "value": v, "unit": "residues/s", "n_gpus": 1,
                      "steps": args.steps, "warmup": max(args.warmup, 2), "higher_is_better": True, "dtype": "u64", "data": "synthetic",
                      "config": {"workload": "c5_sweep", "residues": n_res, "scaled": 1, "k": "5..24",
                                 "moltypes": ["protein", "dayhoff", "hp"]}, "cells": cells}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2_swissprot_hp_k24_s1", choices=sorted(WORKLOADS) + ["c5_sweep"])
    ap.add_argument("--queries", type=int, default=10_000)
    ap.add_argument("--reference-sample", type=int, default=150_000)
    ap.add_argument("--cpu-fast-sample", type=int, default=20_000_000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the target-run and ingest legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps of each leg, write what its last timed step returned (rank 0's index, "
                         "the search leg's pairs and hits, the target run's index) as DIR/<name>.npy in float64: every "
                         "row of a small table, a fixed seeded sample of a large one, and a SHA-256 of every whole "
                         "integer column; the inputs are seeded, so two builds can be compared file by file")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.workload == "c5_sweep" or args.impl == "reference"):
        ap.error("--dump-outputs applies to the GPU index build workloads")
    if args.workload == "c5_sweep":
        return run_c5_sweep(args)
    cfg = WORKLOADS[args.workload]
    if args.impl == "reference":
        return run_reference(args, cfg, args.workload)

    import torch
    import torch.distributed as dist
    import kmerseek_b200 as K
    from kmerseek_b200 import _ffi, shard, synth

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (kmerseek_b200 has no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    comm = shard.Comm(local) if world > 1 else None
    W = max(args.warmup, 3)
    L = _ffi.lib()
    chk = K.errors.check
    dev = torch.device("cuda", local)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(*vals):
        if world == 1:
            return [float(v) for v in vals]
        t = torch.tensor(list(vals), device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t.tolist()]

    def sum_over_ranks(*vals):
        if world == 1:
            return [int(v) for v in vals]
        t = torch.tensor(list(vals), device="cuda", dtype=torch.int64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return [int(x) for x in t.tolist()]

    class Build:
        """One index handle over this rank's shard of a workload's proteome + the timed build loops."""

        def __init__(self, wcfg, res, offs, own_shard=False):
            self.cfg = wcfg
            if own_shard:  # (res, offs) already is this rank's part of the proteome
                sres, soffs, self.bounds = res, offs, None
            else:
                self.bounds = shard.plan_shards(offs, world)
                sres, soffs = shard.shard_of(res, offs, self.bounds, rank)
            self.prot = K.Proteome.from_packed(sres, soffs)
            self.n_res, self.n_prot = self.prot.n_residues, self.prot.n_proteins
            self.idx = K.ProteomeIndex("bench", wcfg["k"], wcfg["scaled"], wcfg["moltype"], device=local)
            self.stream = torch.cuda.ExternalStream(L.ks_index_stream(self.idx._h), device=dev)
            chk(L.ks_index_upload(self.idx._h, self.prot._h))

        def resident(self):
            chk(L.ks_index_clear(self.idx._h))
            chk(L.ks_index_sketch_resident(self.idx._h))
            chk(L.ks_index_finalize(self.idx._h))

        def from_host(self):
            chk(L.ks_index_clear(self.idx._h))
            chk(L.ks_index_add_proteome(self.idx._h, self.prot._h))  # pinned host buffers -> HBM (chunked), overlapped with the sketch
            chk(L.ks_index_finalize(self.idx._h))
            return self.idx.stats()  # the step's result read back on the host

        def timed(self, fn, steps, per_step=None):
            """EXACTLY `steps` calls between barrier + synchronize on both sides; device time by CUDA events on the
            library's stream; max over ranks."""
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(self.stream)
            for _ in range(steps):
                fn()
                if per_step:
                    per_step()
            e1.record(self.stream)
            barrier()
            return max_over_ranks(e0.elapsed_time(e1))[0]

        def close(self):
            self.idx.close()
            self.prot.close()

    # ---- the workload: ONE fixed proteome, sharded by protein over the ranks (strong scaling) ----
    blockwise = "blocks" in cfg
    if blockwise:
        nb_ = cfg["blocks"]
        if nb_ % world:
            raise SystemExit(f"{args.workload}: the rank count must divide {nb_} blocks")
        mine = range(nb_ * rank // world, nb_ * (rank + 1) // world)
        parts = [synth.proteome(cfg["n_residues"] // nb_, cfg["seed"] + i) for i in mine]
        res = np.concatenate([p[0] for p in parts])
        offs = np.concatenate([[0]] + [p[1][1:] + sum(len(q[0]) for q in parts[:j]) for j, p in enumerate(parts)]).astype(np.uint64)
        del parts
        total_res = sum_over_ranks(len(res))[0]
    else:
        res, offs = synth.proteome(cfg["n_residues"], cfg["seed"])
        total_res = int(offs[-1])
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    b = Build(cfg, res, offs, own_shard=blockwise)
    for _ in range(W):
        b.resident()
    st0 = b.idx.stats()
    stage_ms = {"sketch": [], "partition": [], "bucket": [], "csr": []}

    def collect():
        s = b.idx.stats()
        stage_ms["sketch"].append(s["ms_sketch"]); stage_ms["partition"].append(s["ms_sort_partition"])
        stage_ms["bucket"].append(s["ms_sort_bucket"]); stage_ms["csr"].append(s["ms_csr"])

    ms_step = b.timed(b.resident, args.steps, per_step=collect) / args.steps
    st1 = b.idx.stats()
    launches = sum(st1[k] - st0[k] for k in ("sketch_launches", "sort_launches", "csr_launches"))  # this rank, timed region
    value = total_res / (ms_step * 1e-3)

    # ---- e2e: host buffers -> H2D -> build -> stats back, through the public API ----
    for _ in range(2):
        b.from_host()
    ms_e2e = b.timed(b.from_host, args.steps) / args.steps
    e2e_value = total_res / (ms_e2e * 1e-3)
    clocks = sampler.stop() if rank == 0 else None
    st = b.idx.stats()
    dump = {}
    if args.dump_outputs and rank == 0:
        dump.update(dump_index("index_", b.idx))
    n_tuples, n_unique, n_groups = sum_over_ranks(st["n_tuples"], st["n_unique_hashes"], st["n_groups"])
    n_prot_total = sum_over_ranks(len(offs) - 1)[0] if blockwise else len(offs) - 1
    h2d = sum_over_ranks((b.n_res + 7) // 8 * 5 + 72 + (b.n_prot + 1) * 8)[0]
    build_path = st["build_path"]
    stage = {k: max_over_ranks(float(np.mean(v)))[0] for k, v in stage_ms.items()}

    # ---- search leg: BASELINE.json configs[2] -- planted query domains against the same proteome, dayhoff k=16 ----
    if blockwise:
        if dump:
            write_dump(args.dump_outputs, dump)
        return finish_build_only(args, cfg, rank, world, comm, dist if world > 1 else None, peaks, value, ms_step, e2e_value, ms_e2e,
                                 total_res, n_prot_total, n_tuples, n_unique, h2d, build_path, stage, launches, clocks, W)
    scfg = WORKLOADS[SEARCH_WORKLOAD] if cfg["n_residues"] == WORKLOADS[SEARCH_WORKLOAD]["n_residues"] else dict(cfg, k=16, moltype="dayhoff", scaled=1)
    b.close()
    sb = Build(scfg, res, offs)
    sb.resident()
    qres, qoffs, _ = synth.queries(res, offs, args.queries, 77 + 2)  # same seed on every rank: replicated queries
    queries = K.Proteome.from_packed(qres, qoffs)
    q_residues = queries.n_residues
    search = {}
    for label, hits in (("pairs", False), ("pairs_and_hits", True)):
        walls, devs = [], []
        out = None
        for i in range(W + args.steps):
            out = None
            barrier()
            t0 = time.perf_counter()
            out = shard.search_and_gather(sb.idx, queries, comm, pid_base=sb.bounds[rank], hits=hits)
            torch.cuda.synchronize()
            wall = (time.perf_counter() - t0) * 1e3
            wall, = max_over_ranks(wall)
            if i >= W:
                walls.append(wall)
                devs.append(sb.idx.stats()["ms_search"])
        n_pairs = out["n_pairs"] if rank == 0 else 0
        n_hits = len(out["hits"]["hit_qid"]) if (rank == 0 and hits) else 0
        q_hashes = int(out["result"].q_sizes.sum()) if rank == 0 else 0
        alg = search_bytes(q_residues, q_hashes, n_hits, n_pairs)
        wall_ms = float(np.mean(walls))
        dev_ms = max_over_ranks(float(np.mean(devs)))[0]
        search[label] = {"ms_per_batch_wall": wall_ms, "ms_per_batch_kernels": dev_ms, "pairs": int(n_pairs), "hits": int(n_hits),
                         "query_hashes": q_hashes, "algorithmic_bytes": int(alg),
                         "value": q_residues * total_res / (wall_ms * 1e-3)}
        if rank == 0 and label == "pairs":
            keep = {c: out["pairs"][c].copy() for c in ("pair_qid", "pair_pid", "intersect_hashes", "containment")}
        if args.dump_outputs and rank == 0 and hits:
            dump.update(dump_columns("search_", dict(out["pairs"].items())))
            dump.update(dump_columns("search_", dict(out["hits"].items())))
    sb.close()
    verify = None
    if world > 1 and rank == 0:
        # the sharded search against a single-GPU search of the unsharded proteome, at full size
        full = K.ProteomeIndex("verify", scfg["k"], scfg["scaled"], scfg["moltype"], device=local)
        fp = K.Proteome.from_packed(res, offs)
        full.add_proteome(fp)
        full.finalize()
        r1 = K.search(full, queries, hits=False, query_sketches=False)
        verify = {"single_gpu_pairs": int(r1.n_pairs), "sharded_pairs": int(search["pairs"]["pairs"]),
                  "identical": bool(r1.n_pairs == len(keep["pair_qid"]) and all(
                      np.array_equal(r1.pairs[c], keep[c]) for c in keep))}
        full.close()
        fp.close()
        assert verify["identical"], f"sharded search differs from the single-GPU search: {verify}"

    # ---- extra legs (not the headline): the north_star target run, ingest ----
    extra = {}
    if not args.no_extra and args.workload == "c2_swissprot_hp_k24_s1":
        tcfg = WORKLOADS["target_100m_dayhoff_k16_s1"]
        tres, toffs = synth.proteome(tcfg["n_residues"], tcfg["seed"])
        tb = Build(tcfg, tres, toffs)
        for _ in range(W):
            tb.resident()
        t_ms = tb.timed(tb.resident, args.steps) / args.steps
        for _ in range(2):
            tb.from_host()
        t_e2e = tb.timed(tb.from_host, args.steps) / args.steps
        tst = tb.idx.stats()
        if args.dump_outputs and rank == 0:
            dump.update(dump_index("target_index_", tb.idx))
        tt, tu = sum_over_ranks(tst["n_tuples"], tst["n_unique_hashes"])
        tbytes = sketch_bytes(int(toffs[-1]), len(toffs) - 1, tt) + build_bytes(tt, tu)
        extra["target_100m_dayhoff_k16_s1"] = {
            "ms_per_step": t_ms, "value": int(toffs[-1]) / (t_ms * 1e-3), "ms_per_step_e2e": t_e2e,
            "e2e_value": int(toffs[-1]) / (t_e2e * 1e-3), "build_path": BUILD_PATHS[tst["build_path"]],
            "algorithmic_bytes": int(tbytes), "whole_step_frac": tbytes / t_ms / 1e6 / peaks()[0] / world}
        tb.close()
        del tres, toffs
        if rank == 0:
            extra["ingest"] = ingest_leg(K, L, chk, cfg, res, offs, local)

    if rank != 0:
        if comm:
            comm.close()
        if world > 1:
            dist.destroy_process_group()
        return
    if dump:
        write_dump(args.dump_outputs, dump)

    # ---- roofline (SURVEY 8(d) bytes; stage times are CUDA events the library records on its own stream) ----
    peak, peak_src = peaks()
    agg_peak = peak * world  # N GPUs: the job's roofline is N times one GPU's
    sk_b, bd_b = sketch_bytes(total_res, n_prot_total, n_tuples), build_bytes(n_tuples, n_unique)
    build_ms = stage["partition"] + stage["bucket"] + stage["csr"]
    repeat_heavy = n_tuples > 0.25 * {"protein": 20.0, "dayhoff": 6.0, "hp": 2.0}[cfg["moltype"]] ** cfg["k"] / cfg["scaled"]
    if build_path in (1, 2):
        names = {"sketch": "sketch_dense_kernel (ranks + first scatter level)",
                 "partition": "dense_partition_kernel (second scatter level)" if build_path == 1 else "library key sort",
                 "bucket": "dense_bucket_kernel" if build_path == 1 else "dense_count_kernel + dense_write_kernel",
                 "csr": "dir_kernel"}
    else:
        names = {"sketch": "sketch_quad_kernel" + (" (+ first scatter level)" if build_path == 3 else ""),
                 "partition": "pair_partition_kernel (second scatter level)" if build_path == 3 else "partition (library onesweep passes)",
                 "bucket": "bucket_sort_rep_kernel" if repeat_heavy else "bucket_sort_bin_kernel", "csr": "(fused into the bucket kernel)"}
    dom_key = max(("sketch", "bucket"), key=lambda k_: stage[k_])
    dom_bytes = sk_b if dom_key == "sketch" else bd_b
    roof = {
        "bound": "hbm", "kernel": names[dom_key], "achieved": dom_bytes / stage[dom_key] / 1e6, "peak": agg_peak, "unit": "GB/s",
        "frac": dom_bytes / stage[dom_key] / 1e6 / agg_peak,
        "traffic": TRAFFIC_C2.get(names[dom_key]) if (args.workload == "c2_swissprot_hp_k24_s1" and world == 1) else None,
        "peak_source": peak_src + (f" x {world} GPUs" if world > 1 else ""),
        "bytes_model": "SURVEY 8(d): sketch N + 8(P+1) + 16K; index build 24K + 12U + 4 (one logical pass: the partition, bucket "
                       "and directory kernels share it, so the dominant build kernel is charged with all of it); the two "
                       "stages sum to whole_step.algorithmic_bytes",
        "stages": {
            "sketch": {"kernels": names["sketch"], "ms": round(stage["sketch"], 4), "algorithmic_bytes": int(sk_b),
                       "frac": round(sk_b / stage["sketch"] / 1e6 / agg_peak, 4) if stage["sketch"] > 0 else None},
            "index_build": {"kernels": [names["partition"], names["bucket"], names["csr"]],
                            "ms": round(build_ms, 4), "ms_by_kernel": {"partition": round(stage["partition"], 4),
                                                                       "bucket": round(stage["bucket"], 4), "directory": round(stage["csr"], 4)},
                            "algorithmic_bytes": int(bd_b), "frac": round(bd_b / build_ms / 1e6 / agg_peak, 4) if build_ms > 0 else None}},
        "whole_step": {"algorithmic_bytes": int(sk_b + bd_b), "achieved_gbs": (sk_b + bd_b) / ms_step / 1e6,
                       "frac": (sk_b + bd_b) / ms_step / 1e6 / agg_peak}}
    for v in search.values():
        v["roofline"] = {"bound": "hbm", "algorithmic_bytes": v["algorithmic_bytes"], "peak": agg_peak,
                         "frac_kernels": v["algorithmic_bytes"] / v["ms_per_batch_kernels"] / 1e6 / agg_peak if v["ms_per_batch_kernels"] else None,
                         "frac_wall": v["algorithmic_bytes"] / v["ms_per_batch_wall"] / 1e6 / agg_peak,
                         "kernel": "query_kernel",
                         "traffic": TRAFFIC_C3_SEARCH["query_kernel"] if (world == 1 and args.queries == 10_000 and v["hits"] == 0) else None}

    cpu = None
    if not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        vf, dtf, _, _ = cpu_baseline_run(cfg, False, args.cpu_fast_sample, threads)
        v, dt, _, _ = cpu_baseline_run(cfg, True, args.reference_sample, threads)
        cpu = {"value": vf, "unit": "residues/s", "cores": threads, "kind": "port",
               "sample": f"first {args.cpu_fast_sample} residues of the workload, linear-cost variant of the reference's algorithm "
                         f"(binary-search membership, no combined-sketch insert), {dtf:.1f} s",
               "faithful": {"value": v, "unit": "residues/s", "cores": threads,
                            "sample": f"first {args.reference_sample} residues, reference cost structure (two passes, linear "
                                      f"contains, sorted-Vec combined insert; quadratic, so the rate depends on the sample), {dt:.1f} s"}}

    line = {
        "metric": "residues/s sketched+indexed", "value": value, "unit": "residues/s", "n_gpus": world,
        "steps": args.steps, "warmup": W, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": args.workload, "k": cfg["k"], "moltype": cfg["moltype"], "scaled": cfg["scaled"],
                   "residues": total_res, "proteins": n_prot_total, "tuples": n_tuples, "unique_hashes": n_unique,
                   "parallelism": f"one fixed proteome, protein-sharded x{world} (no collective in the build)",
                   "build_path": BUILD_PATHS[build_path],
                   "l2": "inputs (0.2 GB residues, 3 GB tuples over all ranks) exceed the 126 MB L2; no flush needed"},
        "e2e": {"value": e2e_value, "unit": "residues/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": (8 + 16 + 136) * world},
        "gpu_launches": int(launches), "gpu_launches_per_step": int(launches) // args.steps,
        "roofline": roof,
        "cpu_baseline": cpu,
        "search": {"metric": "query x proteome residues/s searched", "workload": SEARCH_WORKLOAD, "unit": "residue pairs/s",
                   "value": search["pairs"]["value"], "queries": args.queries, "query_residues": int(q_residues),
                   "includes": "query H2D, per-query kernels (sketch, lookup, aggregation), scores, "
                               + ("NCCL all-gather + send/recv + merge on rank 0, " if world > 1 else "") + "D2H of the result block",
                   **{k_: v for k_, v in search.items()}, "sharded_equals_single_gpu": verify},
        "extra": extra,
        "clocks": clocks,
    }
    print(json.dumps(line), flush=True)
    if comm:
        comm.close()
    if world > 1:
        dist.destroy_process_group()


def finish_build_only(args, cfg, rank, world, comm, dist, peaks, value, ms_step, e2e_value, ms_e2e, total_res, n_prot, n_tuples,
                      n_unique, h2d, build_path, stage, launches, clocks, W):
    """JSON line of a workload that has build legs only (C4 at full size)."""
    if rank == 0:
        peak, peak_src = peaks()
        agg = peak * world
        sk_b, bd_b = sketch_bytes(total_res, n_prot, n_tuples), build_bytes(n_tuples, n_unique)
        dom = max(("sketch", "bucket"), key=lambda k_: stage[k_])
        dom_b = sk_b if dom == "sketch" else bd_b
        line = {
            "metric": "residues/s sketched+indexed", "value": value, "unit": "residues/s", "n_gpus": world, "steps": args.steps,
            "warmup": W, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u64",
            "data": "synthetic",
            "config": {"workload": args.workload, "k": cfg["k"], "moltype": cfg["moltype"], "scaled": cfg["scaled"],
                       "residues": total_res, "proteins": n_prot, "tuples": n_tuples, "unique_hashes_summed_over_shards": n_unique,
                       "parallelism": f"one fixed proteome of {cfg['blocks']} seeded blocks, protein-sharded x{world}",
                       "build_path": BUILD_PATHS[build_path], "l2": "inputs exceed the 126 MB L2; no flush needed"},
            "e2e": {"value": e2e_value, "unit": "residues/s", "ms_per_step": ms_e2e, "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": (8 + 16 + 136) * world},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": "sketch_quad_kernel" if dom == "sketch" else "bucket sort kernel",
                         "achieved": dom_b / stage[dom] / 1e6, "peak": agg, "unit": "GB/s", "frac": dom_b / stage[dom] / 1e6 / agg,
                         "traffic": None, "peak_source": peak_src + (f" x {world} GPUs" if world > 1 else ""),
                         "stages_ms": {k_: round(v, 4) for k_, v in stage.items()},
                         "whole_step": {"algorithmic_bytes": int(sk_b + bd_b), "frac": (sk_b + bd_b) / ms_step / 1e6 / agg},
                         "note": "scaled = 10: one window in ten becomes a tuple, so the sketch kernel is bound by the hash "
                                 "arithmetic (integer pipe), not by HBM"},
            "cpu_baseline": None, "clocks": clocks}
        print(json.dumps(line), flush=True)
    if comm:
        comm.close()
    if world > 1:
        dist.destroy_process_group()


def ingest_leg(K, L, chk, cfg, res, offs, local):
    """Host-side ingest, timed on rank 0: packed buffers -> pinned ks_proteome, and plain FASTA -> finalized index
    (ks_index_process_fasta = process_fasta, src/rust/index.rs:907-961)."""
    from kmerseek_b200 import synth
    t0 = time.perf_counter()
    p = K.Proteome.from_packed(res, offs)
    t_packed = time.perf_counter() - t0
    p.close()
    d = "/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir()
    path = os.path.join(d, f"ks_bench_{os.getpid()}.fasta")
    try:
        synth.write_fasta(path, res, offs)
        size = os.path.getsize(path)
        best = None
        for _ in range(3):
            idx = K.ProteomeIndex("ingest", cfg["k"], cfg["scaled"], cfg["moltype"], device=local)
            t0 = time.perf_counter()
            chk(L.ks_index_process_fasta(idx._h, path.encode(), 0))
            chk(L.ks_index_sync(idx._h))
            dt = time.perf_counter() - t0
            idx.close()
            best = dt if best is None else min(best, dt)
    finally:
        if os.path.exists(path):
            os.remove(path)
    n = int(offs[-1])
    return {"from_packed_s": t_packed, "from_packed_residues_per_s": n / t_packed,
            "fasta_to_index_s": best, "fasta_to_index_residues_per_s": n / best, "fasta_bytes": size,
            "what": "plain FASTA (60 columns) in " + d + " -> parse, normalise, pack, H2D, sketch, finalize (best of 3)"}


if __name__ == "__main__":
    main()
