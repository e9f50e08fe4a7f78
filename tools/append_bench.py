"""Append against rebuild at C2 size: build C2 (synth.proteome(200 M), hp k24, scaled 1), extend it by batches of 2 M
and 20 M residues with ks_index_append_proteome, and print one JSON line with, per batch size:
  append_ms        wall time of the append call (it returns after its one host read-back), median over --reps
  batch_build_ms   add + finalize of the batch alone on a handle of its own (the append's first half)
  merge_ms         device time of the merge kernels (CUDA events, from the handle's KS_TIMING line)
  merge_bytes      8 n + 4 G + 12 U read for A and for B, written for C; merge_gbps and its fraction of 6 553 GB/s
  rebuild_ms       clear + add(C2) + add(batch) + finalize on one handle: what a caller pays without append
  rebuild_one_batch_ms  clear + add(C2 ++ batch as one proteome) + finalize: a rebuild by a caller who still holds every
                   residue on the host and concatenates them (FASTA parsing not included)
With --profile, one more 2 M append runs under torch.profiler: device time per kernel, and the part of the merge that
compacts segmented inputs (seg_prefix + seg_compact + the directory over A's compacted keys).
Each timed append starts from a freshly built C2 (clear + add + finalize, untimed).  Like bench.py: warm-up runs first,
then the median of the timed runs; the index (GBs) is far larger than L2, so no pass reads from cache.
Usage: python tools/append_bench.py [--reps 5] [--out FILE]"""
import argparse
import json
import os
import re
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

COPY_GBPS = 6553.0  # measured device-to-device copy bandwidth of the B200 (DESIGN.md)
LINE = re.compile(r"\[ks\] append: batch_path (\d+) A_layout (\w+) B_layout (\w+) U_A (\d+) U_B (\d+) matched (\d+) "
                  r"n_C (\d+) batch_ms ([\d.]+) merge_ms ([\d.]+)")


class StderrCapture:
    """The library's KS_TIMING lines go to fd 2: redirect it into a temporary file while a block runs."""

    def __enter__(self):
        self.f = tempfile.TemporaryFile(mode="w+")
        sys.stderr.flush()
        self.saved = os.dup(2)
        os.dup2(self.f.fileno(), 2)
        return self

    def __exit__(self, *a):
        sys.stderr.flush()
        os.dup2(self.saved, 2)
        os.close(self.saved)
        self.f.seek(0)
        self.text = self.f.read()
        self.f.close()


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception:
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--residues", type=int, default=200_000_000)
    ap.add_argument("--batches", default="2000000,20000000")
    ap.add_argument("--out", default=None)
    ap.add_argument("--profile", action="store_true", help="also time each kernel of one 2 M append (torch.profiler)")
    args = ap.parse_args()
    os.environ["KS_TIMING"] = "1"  # read when a handle is created: the merge's device time comes from its line
    import kmerseek_b200 as K
    from kmerseek_b200 import synth

    k, moltype, scaled = 24, "hp", 1
    ra, oa = synth.proteome(args.residues, 20260102)
    a = K.Proteome.from_packed(ra, oa)
    result = {"tool": "append_bench", "gpu": gpu_info(), "c2_residues": args.residues, "k": k, "moltype": moltype,
              "scaled": scaled, "reps": args.reps, "copy_gbps": COPY_GBPS, "batches": []}

    def timed(fn, reps, warmup):
        out = []
        for i in range(warmup + reps):
            t = fn()
            if i >= warmup:
                out.append(t)
        return out

    with K.ProteomeIndex("app", k, scaled, moltype) as idx, K.ProteomeIndex("ref", k, scaled, moltype) as ref, \
            K.ProteomeIndex("bat", k, scaled, moltype) as bat:
        for i, nb in enumerate(int(x) for x in args.batches.split(",")):
            rb, ob = synth.proteome(nb, 4401 + i)
            b = K.Proteome.from_packed(rb, ob)
            ab = K.Proteome.from_packed(np.concatenate([ra, rb]), np.concatenate([oa, ob[1:] + np.uint64(len(ra))]))
            lines, stats_a, stats_c = [], {}, {}

            def one_append():
                idx.clear()
                idx.add_proteome(a)
                idx.finalize()
                stats_a.update(idx.stats())
                with StderrCapture() as cap:
                    t0 = time.perf_counter()
                    idx.append_proteome(b)
                    t1 = time.perf_counter()
                m = LINE.findall(cap.text)
                lines.append(m[-1])
                stats_c.update(idx.stats())
                return (t1 - t0) * 1e3

            app_ms = timed(one_append, args.reps, args.warmup)
            line = lines[-1]
            merge = [float(x[8]) for x in lines[args.warmup:]]

            def one_batch():
                bat.clear()
                t0 = time.perf_counter()
                bat.add_proteome(b)
                bat.finalize()
                bat.stats()  # synchronises
                return (time.perf_counter() - t0) * 1e3

            def one_rebuild():
                t0 = time.perf_counter()
                ref.clear()
                ref.add_proteome(a)
                ref.add_proteome(b)
                ref.finalize()
                ref.stats()
                return (time.perf_counter() - t0) * 1e3

            def one_rebuild_one_batch():
                t0 = time.perf_counter()
                ref.clear()
                ref.add_proteome(ab)
                ref.finalize()
                ref.stats()
                return (time.perf_counter() - t0) * 1e3

            with StderrCapture():
                bat_ms = timed(one_batch, args.reps, args.warmup)
                reb_ms = timed(one_rebuild, args.reps, args.warmup)
                reb1_ms = timed(one_rebuild_one_batch, args.reps, args.warmup)
            ab.close()
            stb = bat.stats()
            sa = stats_a
            side = lambda n, G, U: 8 * n + 4 * G + 12 * U
            model = (side(sa["n_tuples"], sa["n_groups"], sa["n_unique_hashes"]) +
                     side(stb["n_tuples"], stb["n_groups"], stb["n_unique_hashes"]) +
                     side(stats_c["n_tuples"], stats_c["n_groups"], stats_c["n_unique_hashes"]))
            mm = statistics.median(merge)
            result["batches"].append({
                "batch_residues": nb, "batch_path": int(line[0]), "A_layout": line[1], "B_layout": line[2],
                "U_A": int(line[3]), "U_B": int(line[4]), "matched": int(line[5]), "n_C": int(line[6]),
                "append_ms": statistics.median(app_ms), "append_ms_all": app_ms,
                "batch_build_ms": statistics.median(bat_ms), "merge_ms": mm, "merge_ms_all": merge,
                "merge_bytes": model, "merge_gbps": model / (mm * 1e-3) / 1e9,
                "merge_fraction_of_copy": model / (mm * 1e-3) / 1e9 / COPY_GBPS,
                "rebuild_ms": statistics.median(reb_ms), "rebuild_ms_all": reb_ms,
                "rebuild_one_batch_ms": statistics.median(reb1_ms), "rebuild_one_batch_ms_all": reb1_ms,
                "device_bytes_after_append": stats_c["device_bytes"],
            })
        if args.profile:  # one more 2 M append under torch.profiler: device time per merge kernel
            import torch
            from torch.profiler import ProfilerActivity, profile
            b = K.Proteome.from_packed(*synth.proteome(int(args.batches.split(",")[0]), 4401))
            idx.clear()
            idx.add_proteome(a)
            idx.finalize()
            torch.cuda.synchronize()
            with StderrCapture(), profile(activities=[ProfilerActivity.CUDA]) as prof:
                idx.append_proteome(b)
                torch.cuda.synchronize()
            kernels, dir_ms = {}, []
            for e in prof.events():
                if e.device_type.name == "CUDA" and "dir_kernel" in e.name:
                    dir_ms.append(e.device_time_total / 1e3)
            for e in prof.key_averages():
                if e.device_type.name == "CUDA" and e.self_device_time_total > 0:
                    kernels[e.key[:90]] = round(e.self_device_time_total / 1e3, 4)
            result["profile_2m_append_ms"] = dict(sorted(kernels.items(), key=lambda kv: -kv[1])[:16])
            # the directory over A's compacted keys is the first of the append's dir_kernel launches, C's the last
            comp = sum(v for n, v in kernels.items() if "seg_prefix_kernel" in n or "seg_compact_kernel" in n)
            result["profile_2m_compaction_ms"] = round(comp + (dir_ms[0] if len(dir_ms) > 1 else 0.0), 4)
            result["profile_2m_dir_launches_ms"] = [round(x, 4) for x in dir_ms]
    text = json.dumps(result)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
